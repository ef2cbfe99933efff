"""Thin numpy-facing wrapper over the C ABI (one method per ``fyx_*`` entry point).

All compute happens in libfyrox_b200.so's sm_100a kernels; this file only marshals arguments.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib as L


class FyxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"fyx error {code}: {msg}")
        self.code = code


def _u32(a) -> Optional[np.ndarray]:
    if a is None:
        return None
    return np.ascontiguousarray(a, dtype=np.uint32)


def _f32(a) -> Optional[np.ndarray]:
    if a is None:
        return None
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


ANIMATED_VERTEX_LAYOUT = L.fyx_vertex_layout(68, 0, 20, 48, 64)  # scene/mesh/vertex.rs:140-210


def frustum_from_view_projection_matrix(vp) -> Optional[L.fyx_frustum]:
    """Frustum::from_view_projection_matrix (fyrox-math/src/frustum.rs:54-82); None where the reference returns None."""
    lib = L.load()
    m = _f32(np.asarray(vp, dtype=np.float32).reshape(-1))
    assert m.size == 16
    f = L.fyx_frustum()
    rc = lib.fyx_frustum_from_view_projection_matrix(m.ctypes.data_as(L.f32p), C.byref(f))
    return f if rc == 0 else None


def frustum_default() -> L.fyx_frustum:
    f = L.fyx_frustum()
    L.load().fyx_frustum_default(C.byref(f))
    return f


def mat4_mul(a, b) -> np.ndarray:
    """Matrix4 * Matrix4 in nalgebra's order, on 16-float column-major arrays."""
    a = _f32(np.asarray(a).reshape(-1))
    b = _f32(np.asarray(b).reshape(-1))
    out = np.empty(16, dtype=np.float32)
    L.load().fyx_mat4_mul(a.ctypes.data_as(L.f32p), b.ctypes.data_as(L.f32p), out.ctypes.data_as(L.f32p))
    return out


def frustum_to_numpy(f: L.fyx_frustum):
    planes = np.array([[f.planes[p][k] for k in range(4)] for p in range(6)], dtype=np.float32)
    corners = np.array([[f.corners[i][k] for k in range(3)] for i in range(8)], dtype=np.float32)
    return planes, corners


def frustum_from_numpy(planes, corners) -> L.fyx_frustum:
    f = L.fyx_frustum()
    for p in range(6):
        for k in range(4):
            f.planes[p][k] = float(planes[p][k])
    for i in range(8):
        for k in range(3):
            f.corners[i][k] = float(corners[i][k])
    return f


class PinnedBuffer:
    """Page-locked host memory from fyx_host_alloc, viewed as a numpy array."""

    def __init__(self, shape, dtype):
        self._lib = L.load()
        self.dtype = np.dtype(dtype)
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = self._lib.fyx_host_alloc(max(nbytes, 1))
        if not self.ptr:
            raise MemoryError("fyx_host_alloc failed")
        buf = (C.c_char * max(nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            self._lib.fyx_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One fyx_ctx (one GPU)."""

    def __init__(self, device: int = -1, stream: Optional[int] = None):
        self._lib = L.load()
        cfg = L.fyx_config(C.sizeof(L.fyx_config), device, stream, 0)
        h = L.ctx_p()
        rc = self._lib.fyx_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise FyxError(rc, (self._lib.fyx_last_error(None) or b"").decode())
        self._h = h
        self.n_nodes = 0
        self._surfaces = []  # (n_bones, n_verts)

    # -- plumbing --
    def _chk(self, rc: int):
        if rc != 0:
            raise FyxError(rc, (self._lib.fyx_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.fyx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def sync(self):
        self._chk(self._lib.fyx_sync(self._h))

    # -- scene description --
    def set_topology(self, parent, flags=None, render_mask=None, local_aabb=None, root: int = 0, global_index=None):
        parent = _u32(parent)
        n = parent.size
        flags, render_mask, global_index = _u32(flags), _u32(render_mask), _u32(global_index)
        local_aabb = _f32(local_aabb)
        for a, k in ((flags, 1), (render_mask, 1), (global_index, 1), (local_aabb, 6)):
            assert a is None or a.size == n * k
        self._chk(self._lib.fyx_set_topology(self._h, n, root, _ptr(parent), _ptr(flags), _ptr(render_mask), _ptr(local_aabb), _ptr(global_index)))
        self.n_nodes = n

    def set_dfs_order(self, preorder_rank):
        """Pre-order DFS rank of every node (children order of the host graph); None clears it."""
        r = _u32(preorder_rank)
        self._chk(self._lib.fyx_set_dfs_order(self._h, 0 if r is None else r.size, _ptr(r)))

    def set_local_matrices(self, m16, idx=None):
        m16 = _f32(m16)
        idx = _u32(idx)
        count = m16.size // 16
        assert idx is None or idx.size == count
        self._chk(self._lib.fyx_set_local_matrices(self._h, count, _ptr(idx), _ptr(m16)))

    def set_local_trs(self, trs, idx=None):
        """trs: (count, 10) f32 rows of position xyz, rotation quaternion ijkw, scale xyz (fyx_trs)."""
        trs = _f32(trs)
        idx = _u32(idx)
        count = trs.size // 10
        assert idx is None or idx.size == count
        self._chk(self._lib.fyx_set_local_trs(self._h, count, _ptr(idx), _ptr(trs)))

    def set_local_rotations(self, quats, idx=None):
        """quats: (count, 4) f32 unit quaternions i,j,k,w; position/scale stay what the last set_local_trs sent."""
        q = _f32(quats)
        idx = _u32(idx)
        count = q.size // 4
        assert idx is None or idx.size == count
        self._chk(self._lib.fyx_set_local_rotations(self._h, count, _ptr(idx), _ptr(q)))

    def set_transform_statics(self, statics, idx=None):
        """statics: (count, 25) f32 rows: pre_rotation ijkw, post_rotation_matrix (9, column-major), rotation_offset,
        rotation_pivot, scaling_offset, scaling_pivot (fyx_transform_statics)."""
        statics = _f32(statics)
        idx = _u32(idx)
        count = statics.size // 25
        assert idx is None or idx.size == count
        self._chk(self._lib.fyx_set_transform_statics(self._h, count, _ptr(idx), _ptr(statics)))

    def set_flags(self, flags, idx=None):
        flags, idx = _u32(flags), _u32(idx)
        self._chk(self._lib.fyx_set_flags(self._h, flags.size, _ptr(idx), _ptr(flags)))

    def set_render_masks(self, masks, idx=None):
        masks, idx = _u32(masks), _u32(idx)
        self._chk(self._lib.fyx_set_render_masks(self._h, masks.size, _ptr(idx), _ptr(masks)))

    def set_local_aabbs(self, aabbs, idx=None):
        aabbs, idx = _f32(aabbs), _u32(idx)
        self._chk(self._lib.fyx_set_local_aabbs(self._h, aabbs.size // 6, _ptr(idx), _ptr(aabbs)))

    def add_skinned_surface(self, mesh_node: int, bone_nodes, inv_bind_m16, verts=None, layout: L.fyx_vertex_layout = None, n_verts: int = None) -> int:
        bone_nodes = _u32(bone_nodes)
        inv_bind = _f32(inv_bind_m16)
        assert inv_bind.size == bone_nodes.size * 16
        if verts is None:
            n_verts, vptr, lay = 0, None, None
        else:
            lay = layout or ANIMATED_VERTEX_LAYOUT
            if isinstance(verts, np.ndarray):
                verts = np.ascontiguousarray(verts)
                if n_verts is None:
                    n_verts = verts.nbytes // lay.stride
                vptr = verts.ctypes.data_as(C.c_void_p)
            else:  # raw address
                vptr = C.c_void_p(int(verts))
                assert n_verts is not None
        sid = C.c_uint32()
        self._chk(
            self._lib.fyx_add_skinned_surface(
                self._h, mesh_node, bone_nodes.size, _ptr(bone_nodes), _ptr(inv_bind), n_verts, vptr, C.byref(lay) if lay is not None else None, C.byref(sid)
            )
        )
        self._surfaces.append((int(bone_nodes.size), int(n_verts)))
        return sid.value

    def set_blend_shapes(self, surface_id: int, records, weights=None):
        """BlendShapesContainer of a surface: records = uint16 array (n_shapes, layer_stride, 9) of binary16 bit patterns
        (position, normal, tangent offsets per vertex, scene/mesh/surface.rs:92-218); weights = BlendShape::weight (0..100)."""
        r = np.ascontiguousarray(records, dtype=np.uint16)
        if r.size == 0:
            self._chk(self._lib.fyx_set_blend_shapes(self._h, surface_id, 0, None, 0, None))
            return
        assert r.ndim == 3 and r.shape[2] == 9
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float32)
        assert w is None or w.size == r.shape[0]
        self._chk(self._lib.fyx_set_blend_shapes(self._h, surface_id, r.shape[0], r.ctypes.data_as(C.c_void_p), r.shape[1], _ptr(w)))

    def set_skinned_tangents(self, surface_id: int, verts, tangent_offset: int = 32, stride: int = None):
        """Skin the tangents of a surface too (standard.shader:197-200): verts = its VertexBuffer bytes again (tangent = f32 x4 at
        tangent_offset; 32 in AnimatedVertex), stride = bytes per vertex (default: the layout the surface was added with for a
        numpy array of records, else 68); verts may also be a raw (pinned) address.  verts = None turns them off.  Must come before
        set_blend_shapes."""
        if verts is None:
            self._chk(self._lib.fyx_set_skinned_tangents(self._h, surface_id, None, 0, 0))
            return
        if isinstance(verts, np.ndarray):
            verts = np.ascontiguousarray(verts)
            nv = self._surfaces[surface_id][1]
            if stride is None:
                stride = verts.nbytes // nv if nv else ANIMATED_VERTEX_LAYOUT.stride
            assert verts.nbytes >= nv * stride
            vptr = verts.ctypes.data_as(C.c_void_p)
        else:  # raw address of n_verts records
            vptr = C.c_void_p(int(verts))
            stride = ANIMATED_VERTEX_LAYOUT.stride if stride is None else stride
        self._chk(self._lib.fyx_set_skinned_tangents(self._h, surface_id, vptr, stride, tangent_offset))

    def get_skinned_tangents(self, surface_id: int) -> np.ndarray:
        nv = self._surfaces[surface_id][1]
        out = np.empty((nv, 3), dtype=np.float32)
        self._chk(self._lib.fyx_get_skinned_tangents(self._h, surface_id, out.ctypes.data_as(C.c_void_p)))
        return out

    def get_skinned_tangents_device(self, surface_id: int):
        p = C.c_void_p()
        self._chk(self._lib.fyx_get_skinned_tangents_device(self._h, surface_id, C.byref(p)))
        return p.value

    def set_blend_shape_weights(self, surface_id: int, weights):
        w = np.ascontiguousarray(weights, dtype=np.float32)
        self._chk(self._lib.fyx_set_blend_shape_weights(self._h, surface_id, w.size, _ptr(w)))

    def reserve_skinning(self, total_bones: int, total_verts: int):
        self._chk(self._lib.fyx_reserve_skinning(self._h, total_bones, total_verts))

    def commit_surfaces(self):
        self._chk(self._lib.fyx_commit_surfaces(self._h))

    # -- per frame --
    def update_transforms(self, flags: int = L.UPDATE_INCREMENTAL):
        self._chk(self._lib.fyx_update_transforms(self._h, flags))

    @staticmethod
    def _frusta(frusta: Sequence[L.fyx_frustum]):
        arr = (L.fyx_frustum * max(len(frusta), 1))()
        for i, f in enumerate(frusta):
            arr[i] = f
        return arr

    def cull(self, frusta, cam_mask=None, pass_flags=None):
        arr = self._frusta(frusta)
        cm, pf = _u32(cam_mask), _u32(pass_flags)
        self._chk(self._lib.fyx_cull(self._h, len(frusta), arr, _ptr(cm), _ptr(pf)))

    def update_and_cull(self, frusta, update_flags: int = L.UPDATE_INCREMENTAL, cam_mask=None, pass_flags=None):
        arr = self._frusta(frusta)
        cm, pf = _u32(cam_mask), _u32(pass_flags)
        self._chk(self._lib.fyx_update_and_cull(self._h, update_flags, len(frusta), arr, _ptr(cm), _ptr(pf)))

    def get_visible(self, frustum: int = 0, copy: bool = True) -> np.ndarray:
        """Visible node indices of one frustum.  copy=False returns a view of the library's pinned buffer
        (valid until the next cull / frame on this context)."""
        p = L.u32p()
        n = C.c_uint32()
        self._chk(self._lib.fyx_get_visible(self._h, frustum, C.byref(p), C.byref(n)))
        if n.value == 0:
            return np.empty(0, dtype=np.uint32)
        v = np.ctypeslib.as_array(p, shape=(n.value,))
        return v.copy() if copy else v

    def get_visible_device(self, frustum: int = 0):
        d_idx, d_cnt = C.c_void_p(), C.c_void_p()
        self._chk(self._lib.fyx_get_visible_device(self._h, frustum, C.byref(d_idx), C.byref(d_cnt)))
        return d_idx.value, d_cnt.value

    # ---- N4 (LOD filter) ----
    def set_lod_ranges(self, begin_end, idx=None):
        """Per LOD object the [begin, end] of its level (renderer/bundle.rs:898-916); begin NaN removes the node."""
        be = _f32(begin_end)
        ix = _u32(idx)
        self._chk(self._lib.fyx_set_lod_ranges(self._h, be.size // 2, _ptr(ix), _ptr(be)))

    def set_observers(self, observers):
        """observers = [(translation xyz, z_near, z_far), ...], one per frustum of the culls that follow; [] switches LOD off."""
        arr = (L.fyx_observer * max(len(observers), 1))()
        for k, (t, zn, zf) in enumerate(observers):
            arr[k].translation[:] = [float(x) for x in t]
            arr[k].z_near, arr[k].z_far = float(zn), float(zf)
        self._chk(self._lib.fyx_set_observers(self._h, len(observers), C.cast(arr, C.c_void_p)))
        self._n_observers = len(observers)

    # ---- N4 (light list) ----
    def cull_lights(self):
        """Light sources seen by every frustum of the most recent cull (renderer/bundle.rs:926-974)."""
        self._chk(self._lib.fyx_cull_lights(self._h))

    def select_reflection_probes(self) -> np.ndarray:
        """Per observer (set_observers): the reflection probe from_graph would pick (renderer/bundle.rs:918-925), FYX_NONE = none."""
        n = getattr(self, "_n_observers", 0)
        out = np.full(max(n, 1), L.FYX_NONE, np.uint32)
        self._chk(self._lib.fyx_select_reflection_probes(self._h, n, out.ctypes.data_as(C.c_void_p)))
        return out[:n]

    def get_visible_lights(self, frustum: int = 0) -> np.ndarray:
        p = L.u32p()
        n = C.c_uint32()
        self._chk(self._lib.fyx_get_visible_lights(self._h, frustum, C.byref(p), C.byref(n)))
        if n.value == 0:
            return np.empty(0, dtype=np.uint32)
        return np.ctypeslib.as_array(p, shape=(n.value,)).copy()

    # ---- N2: animation sampling on the device ----
    KEY_DTYPE = np.dtype([("location", "<f4"), ("value", "<f4"), ("kind", "<u4"), ("left_tangent", "<f4"), ("right_tangent", "<f4")])
    TRACK_DTYPE = np.dtype([("target_node", "<u4"), ("binding", "<u4"), ("value_kind", "<u4"), ("enabled", "<u4"), ("n_curves", "<u4"),
                            ("first_key", "<u4", 4), ("n_keys", "<u4", 4)])

    def anim_add(self, tracks, keys, speed=1.0, looped=True, time_slice=(0.0, 0.0), time_position=0.0, enabled=True) -> int:
        """Add an Animation (fyrox-animation/src/lib.rs): tracks = TRACK_DTYPE array, keys = KEY_DTYPE array."""
        tracks = np.ascontiguousarray(tracks, dtype=self.TRACK_DTYPE)
        keys = np.ascontiguousarray(keys, dtype=self.KEY_DTYPE)
        d = L.fyx_animation_desc()
        d.struct_size = C.sizeof(L.fyx_animation_desc)
        d.n_tracks, d.tracks = len(tracks), tracks.ctypes.data
        d.n_keys, d.keys = len(keys), keys.ctypes.data
        d.speed, d.time_position = float(speed), float(time_position)
        d.time_slice_start, d.time_slice_end = float(time_slice[0]), float(time_slice[1])
        d.looped, d.enabled = int(bool(looped)), int(bool(enabled))
        out = C.c_uint32()
        self._chk(self._lib.fyx_anim_add(self._h, C.byref(d), C.byref(out)))
        return out.value

    def anim_clear(self):
        self._chk(self._lib.fyx_anim_clear(self._h))

    def anim_set_enabled(self, anim: int, enabled: bool):
        self._chk(self._lib.fyx_anim_set_enabled(self._h, anim, int(bool(enabled))))

    def anim_set_track_enabled(self, anim: int, track: int, enabled: bool):
        self._chk(self._lib.fyx_anim_set_track_enabled(self._h, anim, track, int(bool(enabled))))

    def anim_set_speed(self, anim: int, speed: float):
        self._chk(self._lib.fyx_anim_set_speed(self._h, anim, float(speed)))

    def anim_set_time_position(self, anim: int, t: float):
        self._chk(self._lib.fyx_anim_set_time_position(self._h, anim, float(t)))

    def anim_time_positions(self, first: int, count: int) -> np.ndarray:
        """Animation::time_position() of `count` animations starting at `first` (read back from the device)."""
        out = np.empty(count, dtype=np.float32)
        self._chk(self._lib.fyx_anim_get_time_positions(self._h, first, count, out.ctypes.data_as(C.c_void_p)))
        return out

    def anim_blend_group(self, anims, weights) -> int:
        """BlendAnimations over PlayAnimation sources with constant weights (machine/node/blend.rs:136-166)."""
        a = np.ascontiguousarray(anims, dtype=np.uint32)
        w = np.ascontiguousarray(weights, dtype=np.float32)
        assert a.size == w.size
        out = C.c_uint32()
        self._chk(self._lib.fyx_anim_blend_group(self._h, a.size, _ptr(a), _ptr(w), C.byref(out)))
        return out.value

    def anim_set_blend_weights(self, group: int, weights):
        w = np.ascontiguousarray(weights, dtype=np.float32)
        self._chk(self._lib.fyx_anim_set_blend_weights(self._h, group, w.size, _ptr(w)))

    def animate(self, dt: float):
        """AnimationContainer::update_animations(dt) for every animation (scene/animation/mod.rs:83-88)."""
        self._chk(self._lib.fyx_animate(self._h, float(dt)))

    # ---- N3: draw-prep after the cull ----
    def set_bundle_ids(self, ids, idx=None):
        """Per-node bundle id = dense id of the (material, surface data, render path) key of
        RenderDataBundleStorage::push (renderer/bundle.rs:1253-1257)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        ix = _u32(idx)
        self._chk(self._lib.fyx_set_bundle_ids(self._h, len(ids), _ptr(ix), _ptr(ids)))

    def set_node_surfaces(self, nodes, surfaces):
        """Mesh::surfaces of the given nodes: surfaces[i] = list of (bundle_id, skin_surface_id or None) for node nodes[i]."""
        idx = np.ascontiguousarray(nodes, dtype=np.uint32)
        first = np.zeros(len(idx) + 1, np.uint32)
        b, sk = [], []
        for i, lst in enumerate(surfaces):
            for bid, sid in lst:
                b.append(bid)
                sk.append(L.FYX_NONE if sid is None else sid)
            first[i + 1] = len(b)
        ba = np.ascontiguousarray(b, dtype=np.uint32)
        sa = np.ascontiguousarray(sk, dtype=np.uint32)
        self._chk(self._lib.fyx_set_node_surfaces(self._h, len(idx), _ptr(idx), _ptr(first), ba.ctypes.data_as(C.c_void_p) if ba.size else None,
                                                  sa.ctypes.data_as(C.c_void_p) if sa.size else None))

    def get_instance_surfaces(self, frustum: int, count: int) -> np.ndarray:
        p = L.u32p()
        self._chk(self._lib.fyx_get_instance_surfaces(self._h, frustum, C.byref(p)))
        return np.ctypeslib.as_array(p, shape=(count,)).copy() if count else np.empty(0, np.uint32)

    def enable_instances(self, enable: bool = True):
        self._chk(self._lib.fyx_enable_instances(self._h, 1 if enable else 0))

    def pack_instances(self, frustum: int, view_m16, view_projection_m16) -> dict:
        """Instances of the frustum's visible list grouped by bundle: dict with node (u32[n]), sort_index (u64[n]),
        world / wvp (f32[n,16], column-major) and bundles (structured array: id, first, count, sort_index)."""
        v = np.ascontiguousarray(view_m16, dtype=np.float32).reshape(16)
        vp = np.ascontiguousarray(view_projection_m16, dtype=np.float32).reshape(16)
        self._chk(self._lib.fyx_pack_instances(self._h, frustum, _ptr(v), _ptr(vp)))
        out = L.fyx_instances()
        self._chk(self._lib.fyx_get_instances(self._h, frustum, C.byref(out)))
        n, nb = out.count, out.n_bundles
        bdt = np.dtype([("id", "<u4"), ("first", "<u4"), ("count", "<u4"), ("reserved", "<u4"), ("sort_index", "<u8")])

        def arr(p, dtype, count):
            if count == 0:
                return np.empty(0, dtype=dtype)
            buf = (C.c_char * (count * np.dtype(dtype).itemsize)).from_address(p)
            return np.frombuffer(buf, dtype=dtype, count=count).copy()

        mats = arr(out.matrices, np.float32, n * 32).reshape(n, 2, 16)
        return {
            "surface": self.get_instance_surfaces(frustum, n),
            "node": arr(out.node, np.uint32, n),
            "sort_index": arr(out.sort_index, np.uint64, n),
            "world": mats[:, 0, :].copy(),
            "wvp": mats[:, 1, :].copy(),
            "bundles": arr(out.bundles, bdt, nb),
        }

    def pack_bone_matrices(self, frustum: int):
        """Bone-matrix blocks (255 mat4, zero padded) of the skinned instances of the last pack_instances (bundle.rs:484-496)."""
        self._chk(self._lib.fyx_pack_bone_matrices(self._h, frustum))

    def get_bone_matrix_block(self, frustum: int, instance: int):
        """(255,16) f32 block of packed instance `instance`, or None for an unskinned instance."""
        out = np.empty((255, 16), dtype=np.float32)
        has = C.c_uint32()
        self._chk(self._lib.fyx_get_bone_matrix_block(self._h, frustum, instance, out.ctypes.data_as(C.c_void_p), C.byref(has)))
        return out if has.value else None

    def build_palettes(self):
        self._chk(self._lib.fyx_build_palettes(self._h))

    def skin(self):
        self._chk(self._lib.fyx_skin(self._h))

    def render_prep(self, *, update_flags=L.UPDATE_INCREMENTAL, changed_m16=None, changed_trs=None, changed_rot=None, changed_idx=None, n_changed=None, frusta=(), cam_mask=None,
                    pass_flags=None, do_palettes=True, do_skin=True, readback_visible=True, async_=False, allgather=False,
                    animate_dt=None, readback_own=False):
        """One frame (fyx_render_prep). changed_m16 / changed_idx may be numpy arrays or raw (pinned) addresses."""
        d = L.fyx_frame_desc()
        d.struct_size = C.sizeof(L.fyx_frame_desc)
        d.update_flags = update_flags
        keep = []
        if changed_rot is not None:
            payload, width, field = changed_rot, 4, "changed_rot"
        elif changed_trs is not None:
            payload, width, field = changed_trs, 10, "changed_trs"
        else:
            payload, width, field = changed_m16, 16, "changed_m16"
        if payload is not None:
            if isinstance(payload, np.ndarray):
                m = _f32(payload)
                keep.append(m)
                setattr(d, field, m.ctypes.data)
                d.n_changed = m.size // width if n_changed is None else n_changed
            else:
                setattr(d, field, int(payload))
                d.n_changed = int(n_changed)
            if changed_idx is not None:
                if isinstance(changed_idx, np.ndarray):
                    ix = _u32(changed_idx)
                    keep.append(ix)
                    d.changed_idx = ix.ctypes.data
                else:
                    d.changed_idx = int(changed_idx)
        arr = self._frusta(frusta)
        d.n_frusta = len(frusta)
        d.frusta = C.cast(arr, C.POINTER(L.fyx_frustum))
        cm, pf = _u32(cam_mask), _u32(pass_flags)
        keep += [cm, pf, arr]
        d.cam_mask = None if cm is None else cm.ctypes.data
        d.pass_flags = None if pf is None else pf.ctypes.data
        d.do_palettes = 1 if do_palettes else 0
        d.do_skin = 1 if do_skin else 0
        d.readback_visible = 1 if readback_visible else 0
        d.flags = (L.FRAME_ASYNC if async_ else 0) | (L.FRAME_ALLGATHER if allgather else 0) | (L.FRAME_READBACK_OWN if readback_own else 0)
        if animate_dt is not None:
            d.do_animate = 1
            d.animate_dt = float(animate_dt)
        if async_:
            self._async_keep = keep  # inputs must outlive the enqueued frame
        self._chk(self._lib.fyx_render_prep(self._h, C.byref(d)))

    def frame_wait(self):
        """Collect the oldest pipelined (async + read-back) frame; its visible lists become readable."""
        self._chk(self._lib.fyx_frame_wait(self._h))

    # -- read-back --
    def _gather(self, fn, idx, count, width, dtype):
        idx = _u32(idx)
        n = self.n_nodes if idx is None and count is None else (idx.size if idx is not None else count)
        out = np.empty((n, width) if width > 1 else (n,), dtype=dtype)
        self._chk(fn(self._h, n, _ptr(idx), out.ctypes.data_as(C.c_void_p)))
        return out

    def get_global_matrices(self, idx=None, count=None) -> np.ndarray:
        return self._gather(self._lib.fyx_get_global_matrices, idx, count, 16, np.float32)

    def get_world_aabbs(self, idx=None, count=None) -> np.ndarray:
        return self._gather(self._lib.fyx_get_world_aabbs, idx, count, 6, np.float32)

    def get_global_flags(self, idx=None, count=None) -> np.ndarray:
        return self._gather(self._lib.fyx_get_global_flags, idx, count, 1, np.uint32)

    def get_palette(self, surface_id: int) -> np.ndarray:
        nb = self._surfaces[surface_id][0]
        out = np.empty((nb, 16), dtype=np.float32)
        self._chk(self._lib.fyx_get_palette(self._h, surface_id, out.ctypes.data_as(C.c_void_p)))
        return out

    def get_skinned(self, surface_id: int, normals: bool = True):
        nv = self._surfaces[surface_id][1]
        pos = np.empty((nv, 3), dtype=np.float32)
        nrm = np.empty((nv, 3), dtype=np.float32) if normals else None
        self._chk(self._lib.fyx_get_skinned(self._h, surface_id, pos.ctypes.data_as(C.c_void_p), None if nrm is None else nrm.ctypes.data_as(C.c_void_p)))
        return pos, nrm

    def get_skinned_device(self, surface_id: int):
        p, n = C.c_void_p(), C.c_void_p()
        self._chk(self._lib.fyx_get_skinned_device(self._h, surface_id, C.byref(p), C.byref(n)))
        return p.value, n.value

    def timings(self) -> dict:
        t = L.fyx_timings()
        self._chk(self._lib.fyx_get_timings(self._h, C.byref(t)))
        return {n: getattr(t, n) for n, _ in L.fyx_timings._fields_}

    def kernel_launch_count(self) -> int:
        return int(self._lib.fyx_kernel_launch_count(self._h))

    # -- multi-GPU --
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        lib = L.load()
        rc = lib.fyx_comm_get_unique_id(buf)
        if rc != 0:
            raise FyxError(rc, (lib.fyx_last_error(None) or b"").decode())
        return buf.raw

    def comm_init(self, nranks: int, rank: int, uid: bytes):
        assert len(uid) == 128
        self._chk(self._lib.fyx_comm_init(self._h, nranks, rank, C.create_string_buffer(uid, 128)))

    def comm_mode(self) -> str:
        """How the visible lists are exchanged (fyx_comm_mode): decided collectively at the first gathered frame."""
        m = int(self._lib.fyx_comm_mode(self._h))
        if not m:
            return "none"
        if m & L.COMM_UNDECIDED:
            return "nccl initialised, exchange not built yet"
        dev = "peer stores over NVLink (cudaIpc)" if m & L.COMM_PEER_STORES else "ncclAllGather (counts, padded slots, pack kernels)"
        host = "node-wide host segment (each rank copies its own lists)" if m & L.COMM_HOST_SEGMENT else "private copy of the gathered device lists per rank"
        return f"device: {dev}; host: {host}"

    def comm_stats(self) -> dict:
        """The most recent exchange of this rank: entries, NVLink egress bytes, device time (fyx_comm_get_stats)."""
        st = L.fyx_comm_stats()
        self._chk(self._lib.fyx_comm_get_stats(self._h, C.byref(st)))
        return {n: getattr(st, n) for n, _ in L.fyx_comm_stats._fields_}

    def allgather_visible(self):
        self._chk(self._lib.fyx_allgather_visible(self._h))

    def get_visible_gathered(self, frustum: int = 0, copy: bool = True) -> np.ndarray:
        p = L.u32p()
        n = C.c_uint32()
        self._chk(self._lib.fyx_get_visible_gathered(self._h, frustum, C.byref(p), C.byref(n)))
        if n.value == 0:
            return np.empty(0, dtype=np.uint32)
        v = np.ctypeslib.as_array(p, shape=(n.value,))
        return v.copy() if copy else v

    def get_visible_gathered_device(self, frustum: int = 0):
        p = C.c_void_p()
        n = C.c_uint32()
        self._chk(self._lib.fyx_get_visible_gathered_device(self._h, frustum, C.byref(p), C.byref(n)))
        return p.value, n.value
