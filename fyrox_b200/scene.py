"""Host-side mirror of the reference's interface for the render-prep path.

The reference is Rust and this image has no Rust toolchain, so the host side above the C ABI is
written in Python with the reference's names and argument meaning, so that the parity tests read
like the reference's own tests:

    Handle, Pool numbering          fyrox-core/src/pool/handle.rs:38-47, pool/mod.rs
    Transform / TransformBuilder    fyrox-impl/src/scene/transform.rs:79-127,421-550
    Base fields on Node             fyrox-impl/src/scene/base.rs:389-483
    Graph::{new,add_node,link_nodes,remove_node,update,update_hierarchical_data,global_scale}
                                    fyrox-impl/src/scene/graph/mod.rs:408-424,1272-1292,1459-1504,1835-1845,2044-2131
    ObserverPosition                fyrox-impl/src/renderer/observer.rs:47-60
    RenderDataBundleStorage::from_graph   fyrox-impl/src/renderer/bundle.rs:873-1009

What a Rust shim would do at S1/S2/S3 (SURVEY §8b) is what `Graph.update` / `from_graph` do here:
scatter changed properties through the C ABI, then run the sm_100a kernels.  No arithmetic of the hot
path happens in this file except `Transform.matrix()` (the reference computes it on the host too).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np

from . import _lib as L
from .context import ANIMATED_VERTEX_LAYOUT, Context, frustum_default, frustum_from_view_projection_matrix, mat4_mul

f32 = np.float32


@dataclass(frozen=True)
class Handle:
    """Handle<Node>{index, generation} (fyrox-core/src/pool/handle.rs:38-47)."""

    index: int = 0
    generation: int = 0

    def is_none(self) -> bool:
        return self.generation == 0

    def is_some(self) -> bool:
        return self.generation != 0


Handle.NONE = Handle(0, 0)


def _quat_to_rotation_matrix(q) -> List[np.float32]:
    """UnitQuaternion::to_rotation_matrix, column-major 3x3 (nalgebra)."""
    i, j, k, w = (f32(x) for x in q)
    two = f32(2.0)
    ww, ii, jj, kk = w * w, i * i, j * j, k * k
    ij, wk, wj = i * j * two, w * k * two, w * j * two
    ik, jk, wi = i * k * two, j * k * two, w * i * two
    m11, m12, m13 = ww + ii - jj - kk, ij - wk, wj + ik
    m21, m22, m23 = wk + ij, ww - ii + jj - kk, jk - wi
    m31, m32, m33 = ik - wj, wi + jk, ww - ii - jj + kk
    return [m11, m21, m31, m12, m22, m32, m13, m23, m33]


class Transform:
    """Transform (scene/transform.rs:79-127): TRS + FBX-style pivots/offsets, cached local matrix."""

    def __init__(self):
        self.local_position = np.zeros(3, f32)
        self.local_rotation = np.array([0, 0, 0, 1], f32)  # i, j, k, w
        self.local_scale = np.ones(3, f32)
        self.pre_rotation = np.array([0, 0, 0, 1], f32)
        self.post_rotation_matrix = np.eye(3, dtype=f32).T.reshape(9).copy()  # cached inverse (transform.rs:160-172)
        self.rotation_offset = np.zeros(3, f32)
        self.rotation_pivot = np.zeros(3, f32)
        self.scaling_offset = np.zeros(3, f32)
        self.scaling_pivot = np.zeros(3, f32)
        self._matrix = None
        self._on_change = None

    # setters mark dirty and notify (TrackedProperty::deref_mut, base.rs:343-352)
    def _touch(self):
        self._matrix = None
        if self._on_change:
            self._on_change()

    def set_position(self, v):
        self.local_position = np.asarray(v, f32)
        self._touch()
        return self

    def set_rotation(self, q):
        self.local_rotation = np.asarray(q, f32)
        self._touch()
        return self

    def set_scale(self, v):
        self.local_scale = np.asarray(v, f32)
        self._touch()
        return self

    def position(self):
        return self.local_position

    def scale(self):
        return self.local_scale

    def matrix(self) -> np.ndarray:
        """Transform::matrix / calculate_local_transform (transform.rs:421-550), f32 op by op."""
        if self._matrix is not None:
            return self._matrix
        por = [f32(x) for x in self.post_rotation_matrix]
        pr = _quat_to_rotation_matrix(self.pre_rotation)
        r = _quat_to_rotation_matrix(self.local_rotation)
        sx, sy, sz = (f32(x) for x in self.local_scale)
        tx, ty, tz = (f32(x) for x in self.local_position)
        rpx, rpy, rpz = (f32(x) for x in self.rotation_pivot)
        rox, roy, roz = (f32(x) for x in self.rotation_offset)
        spx, spy, spz = (f32(x) for x in self.scaling_pivot)
        sox, soy, soz = (f32(x) for x in self.scaling_offset)
        a0 = pr[0] * r[0] + pr[3] * r[1] + pr[6] * r[2]
        a1 = pr[1] * r[0] + pr[4] * r[1] + pr[7] * r[2]
        a2 = pr[2] * r[0] + pr[5] * r[1] + pr[8] * r[2]
        a3 = pr[0] * r[3] + pr[3] * r[4] + pr[6] * r[5]
        a4 = pr[1] * r[3] + pr[4] * r[4] + pr[7] * r[5]
        a5 = pr[2] * r[3] + pr[5] * r[4] + pr[8] * r[5]
        a6 = pr[0] * r[6] + pr[3] * r[7] + pr[6] * r[8]
        a7 = pr[1] * r[6] + pr[4] * r[7] + pr[7] * r[8]
        a8 = pr[2] * r[6] + pr[5] * r[7] + pr[8] * r[8]
        f0 = por[0] * a0 + por[1] * a3 + por[2] * a6
        f1 = por[0] * a1 + por[1] * a4 + por[2] * a7
        f2 = por[0] * a2 + por[1] * a5 + por[2] * a8
        f3 = por[3] * a0 + por[4] * a3 + por[5] * a6
        f4 = por[3] * a1 + por[4] * a4 + por[5] * a7
        f5 = por[3] * a2 + por[4] * a5 + por[5] * a8
        f6 = por[6] * a0 + por[7] * a3 + por[8] * a6
        f7 = por[6] * a1 + por[7] * a4 + por[8] * a7
        f8 = por[6] * a2 + por[7] * a5 + por[8] * a8
        z = f32(0.0)
        m0, m1, m2, m3 = sx * f0, sx * f1, sx * f2, z
        m4, m5, m6, m7 = sy * f3, sy * f4, sy * f5, z
        m8, m9, m10, m11 = sz * f6, sz * f7, sz * f8, z
        k0, k1, k2 = spx * f0, spy * f3, spz * f6
        m12 = rox + rpx + tx - rpx * f0 - rpy * f3 - rpz * f6 + sox * f0 + k0 + soy * f3 + k1 + soz * f6 + k2 - sx * k0 - sy * k1 - sz * k2
        k3, k4, k5 = spx * f1, spy * f4, spz * f7
        m13 = roy + rpy + ty - rpx * f1 - rpy * f4 - rpz * f7 + sox * f1 + k3 + soy * f4 + k4 + soz * f7 + k5 - sx * k3 - sy * k4 - sz * k5
        k6, k7, k8 = spx * f2, spy * f5, spz * f8
        m14 = roz + rpz + tz - rpx * f2 - rpy * f5 - rpz * f8 + sox * f2 + k6 + soy * f5 + k7 + soz * f8 + k8 - sx * k6 - sy * k7 - sz * k8
        self._matrix = np.array([m0, m1, m2, m3, m4, m5, m6, m7, m8, m9, m10, m11, m12, m13, m14, f32(1.0)], dtype=f32)
        return self._matrix


class TransformBuilder:
    def __init__(self):
        self._t = Transform()

    def with_local_position(self, v):
        self._t.local_position = np.asarray(v, f32)
        return self

    def with_local_rotation(self, q):
        self._t.local_rotation = np.asarray(q, f32)
        return self

    def with_local_scale(self, v):
        self._t.local_scale = np.asarray(v, f32)
        return self

    def build(self) -> Transform:
        return self._t


@dataclass
class BlendShape:
    """BlendShape (scene/mesh/surface.rs:71-90): weight in 0..100 (default 100) and a name."""

    weight: float = 100.0
    name: str = ""


@dataclass
class BlendShapesContainer:
    """BlendShapesContainer (scene/mesh/surface.rs:92-218): the shapes and the volume texture from_lists packs them into —
    here as its texels: uint16 (n_shapes, width * height, 9) binary16 patterns (position, normal, tangent offsets)."""

    blend_shapes: List[BlendShape] = field(default_factory=list)
    blend_shape_storage: Optional[np.ndarray] = None


class BatchingMode:
    """BatchingMode (scene/mesh/mod.rs:120-140)."""

    NONE, STATIC, DYNAMIC = "None", "Static", "Dynamic"


@dataclass
class Surface:
    """Surface (scene/mesh/surface.rs:1249-1271): bone handles + the VertexBuffer bytes (+ SurfaceData::blend_shapes_container)."""

    bones: List[Handle] = field(default_factory=list)
    vertex_buffer: Optional[np.ndarray] = None  # uint8, AnimatedVertex records
    surface_id: Optional[int] = None            # fyx surface id once uploaded
    blend_shapes_container: Optional[BlendShapesContainer] = None
    skin_tangents: bool = False                 # also skin the tangents (fyx_set_skinned_tangents) for a normal-mapped renderer
    _shapes_uploaded: bool = False


class Node:
    """Base (scene/base.rs:389-483) plus the Mesh bits on the path (scene/mesh/mod.rs:328-377)."""

    def __init__(self, kind: str = "pivot", name: str = ""):
        self.kind = kind  # "pivot" | "mesh"
        self.name = name
        self._local_transform = Transform()
        self._visibility = True
        self._enabled = True
        self.frustum_culling = True
        self.cast_shadows = True
        self.render_mask = 0xFFFFFFFF
        self.parent = Handle.NONE
        self.children: List[Handle] = []
        self.inv_bind_pose_transform = np.eye(4, dtype=f32).T.reshape(16).copy()
        self.local_bounding_box = np.array([-0.5, -0.5, -0.5, 0.5, 0.5, 0.5], f32) if kind != "mesh" else np.array(
            [np.finfo(f32).max] * 3 + [-np.finfo(f32).max] * 3, f32)
        self.surfaces: List[Surface] = []
        self.batching_mode = BatchingMode.NONE  # Mesh::batching_mode (scene/mesh/mod.rs:372)
        self._graph: Optional["Graph"] = None
        self._handle = Handle.NONE

    # Mesh::blend_shapes / blend_shapes_mut (scene/mesh/mod.rs:449-456): the weights the renderer divides by 100 (:794-798)
    def blend_shapes(self) -> List[BlendShape]:
        for s in self.surfaces:
            if s.blend_shapes_container is not None:
                return s.blend_shapes_container.blend_shapes
        return []

    def blend_shapes_mut(self) -> List[BlendShape]:
        self._notify("blend_shapes")
        return self.blend_shapes()

    def set_batching_mode(self, mode: str):
        """Mesh::set_batching_mode (scene/mesh/mod.rs:612-617); Static => RdcControlFlow::Break when the mesh is rendered."""
        self.batching_mode = mode
        self._notify("flags")

    # tracked properties
    def local_transform(self) -> Transform:
        return self._local_transform

    def local_transform_mut(self) -> Transform:
        self._notify("transform")
        self._local_transform._matrix = self._local_transform._matrix  # caller mutates through setters
        return self._local_transform

    def set_local_transform(self, t: Transform):
        self._local_transform = t
        t._on_change = lambda: self._notify("transform")
        self._notify("transform")

    def visibility(self) -> bool:
        return self._visibility

    def set_visibility(self, v: bool):
        self._visibility = bool(v)
        self._notify("flags")

    def is_enabled(self) -> bool:
        return self._enabled

    def set_enabled(self, v: bool):
        self._enabled = bool(v)
        self._notify("flags")

    def set_frustum_culling(self, v: bool):
        self.frustum_culling = bool(v)
        self._notify("flags")

    def set_cast_shadows(self, v: bool):
        self.cast_shadows = bool(v)
        self._notify("flags")

    def set_render_mask(self, m: int):
        self.render_mask = int(m) & 0xFFFFFFFF
        self._notify("mask")

    def set_local_bounding_box(self, aabb6):
        self.local_bounding_box = np.asarray(aabb6, f32)
        self._notify("aabb")

    def _notify(self, what: str):
        if self._graph is not None:
            self._graph._mark(self._handle, what)

    # hierarchical values (valid after Graph.update)
    def global_transform(self) -> np.ndarray:
        return self._graph._global_matrix(self._handle)

    def global_position(self) -> np.ndarray:
        return self.global_transform()[12:15]

    def global_visibility(self) -> bool:
        return bool(self._graph._global_flags(self._handle) & L.NODE_GLOBAL_VISIBILITY)

    def is_globally_enabled(self) -> bool:
        return bool(self._graph._global_flags(self._handle) & L.NODE_GLOBAL_ENABLED)

    def world_bounding_box(self) -> np.ndarray:
        return self._graph._world_aabb(self._handle)

    def flags_word(self) -> int:
        f = L.NODE_ALIVE
        f |= L.NODE_VISIBILITY if self._visibility else 0
        f |= L.NODE_ENABLED if self._enabled else 0
        f |= L.NODE_FRUSTUM_CULLING if self.frustum_culling else 0
        f |= L.NODE_CAST_SHADOWS if self.cast_shadows else 0
        f |= L.NODE_RENDERABLE if self.kind == "mesh" else 0
        f |= L.NODE_STATIC_BATCH if (self.kind == "mesh" and self.batching_mode == BatchingMode.STATIC) else 0
        return f


class BaseBuilder:
    """BaseBuilder/PivotBuilder/MeshBuilder folded into one (scene/base.rs:1255-1400)."""

    def __init__(self, kind: str = "pivot"):
        self._n = Node(kind)
        self._children: List[Handle] = []

    def with_local_transform(self, t: Transform):
        self._n._local_transform = t
        return self

    def with_visibility(self, v: bool):
        self._n._visibility = bool(v)
        return self

    def with_enabled(self, v: bool):
        self._n._enabled = bool(v)
        return self

    def with_frustum_culling(self, v: bool):
        self._n.frustum_culling = bool(v)
        return self

    def with_cast_shadows(self, v: bool):
        self._n.cast_shadows = bool(v)
        return self

    def with_render_mask(self, m: int):
        self._n.render_mask = int(m)
        return self

    def with_local_bounding_box(self, aabb6):
        self._n.local_bounding_box = np.asarray(aabb6, f32)
        return self

    def with_inv_bind_pose_transform(self, m16):
        self._n.inv_bind_pose_transform = np.asarray(m16, f32).reshape(16)
        return self

    def with_surfaces(self, surfaces: List[Surface]):
        self._n.surfaces = list(surfaces)
        return self

    def with_child(self, h: Handle):
        self._children.append(h)
        return self

    def with_children(self, hs):
        self._children.extend(hs)
        return self

    def build(self, graph: "Graph") -> Handle:
        h = graph.add_node(self._n)
        for c in self._children:
            graph.link_nodes(c, h)
        return h


def PivotBuilder(base: BaseBuilder = None) -> BaseBuilder:
    b = base or BaseBuilder()
    b._n.kind = "pivot"
    return b


def MeshBuilder(base: BaseBuilder = None) -> BaseBuilder:
    b = base or BaseBuilder()
    b._n.kind = "mesh"
    if np.all(b._n.local_bounding_box == np.array([-0.5, -0.5, -0.5, 0.5, 0.5, 0.5], f32)):
        b._n.local_bounding_box = np.array([np.finfo(f32).max] * 3 + [-np.finfo(f32).max] * 3, f32)
    return b


class Graph:
    """Graph (scene/graph/mod.rs:130-175): a pool of nodes; hierarchical data lives on the GPU."""

    def __init__(self, ctx: Optional[Context] = None):
        self.ctx = ctx or Context()
        self._records: List[Optional[Node]] = []
        self._generation: List[int] = []
        self._free: List[int] = []
        self.root = Handle.NONE
        self._topology_dirty = True
        self._dirty: Dict[str, set] = {"transform": set(), "flags": set(), "mask": set(), "aabb": set(), "blend_shapes": set()}
        self._cache: Dict[str, np.ndarray] = {}
        self._surfaces_uploaded = 0
        self.root = self.add_node(Node("pivot", "__ROOT__"))  # Graph::new, graph/mod.rs:408-424

    # ---- pool ----
    def capacity(self) -> int:
        return len(self._records)

    def is_valid_handle(self, h: Handle) -> bool:
        return h.is_some() and h.index < len(self._records) and self._records[h.index] is not None and self._generation[h.index] == h.generation

    def try_get_node(self, h: Handle) -> Optional[Node]:
        return self._records[h.index] if self.is_valid_handle(h) else None

    def __getitem__(self, h: Handle) -> Node:
        n = self.try_get_node(h)
        if n is None:
            raise KeyError(f"invalid handle {h}")
        return n

    def add_node(self, node: Node) -> Handle:
        """Graph::add_node (graph/mod.rs:2044-2088): spawn, link to the root, notify."""
        if self._free:
            i = self._free.pop()
            self._generation[i] += 1
            self._records[i] = node
        else:
            i = len(self._records)
            self._records.append(node)
            self._generation.append(1)
        h = Handle(i, self._generation[i])
        node._graph, node._handle = self, h
        node._local_transform._on_change = lambda: node._notify("transform")
        for s in node.surfaces:
            s.surface_id = None
        self._topology_dirty = True
        if self.root.is_none():
            self.root = h
        else:
            self.link_nodes(h, self.root)
        return h

    def link_nodes(self, child: Handle, parent: Handle):
        """Graph::link_nodes (graph/mod.rs:2114-2131)."""
        self._isolate(child)
        self[child].parent = parent
        self[parent].children.append(child)
        self._topology_dirty = True

    def _isolate(self, h: Handle):
        n = self[h]
        p = self.try_get_node(n.parent)
        n.parent = Handle.NONE
        if p is not None and h in p.children:
            p.children.remove(h)

    def remove_node(self, h: Handle):
        """Graph::remove_node (graph/mod.rs:2091-2111): frees the whole sub-tree."""
        self._isolate(h)
        stack = [h]
        while stack:
            x = stack.pop()
            n = self.try_get_node(x)
            if n is None:
                continue
            stack.extend(n.children)
            self._records[x.index] = None
            self._free.append(x.index)
        self._topology_dirty = True

    def _mark(self, h: Handle, what: str):
        self._dirty[what].add(h.index)
        self._cache.clear()

    # ---- sync + update ----
    def _sync(self):
        cap = len(self._records)
        if self._topology_dirty:
            parent = np.full(cap, L.FYX_NONE, np.uint32)
            flags = np.zeros(cap, np.uint32)
            mask = np.zeros(cap, np.uint32)
            aabb = np.zeros((cap, 6), f32)
            local = np.zeros((cap, 16), f32)
            for i, n in enumerate(self._records):
                if n is None:
                    continue
                p = self.try_get_node(n.parent)
                parent[i] = n.parent.index if p is not None else L.FYX_NONE
                flags[i] = n.flags_word()
                mask[i] = n.render_mask
                aabb[i] = n.local_bounding_box
                local[i] = n.local_transform().matrix()
            self.ctx.set_topology(parent, flags, mask, aabb, root=self.root.index)
            alive = np.nonzero(flags & L.NODE_ALIVE)[0].astype(np.uint32)
            if alive.size:
                self.ctx.set_local_matrices(local[alive], alive)
            # surfaces refer to node indices: (re)upload all of them after a topology change
            self._upload_surfaces(reset=True)
            self._topology_dirty = False
            for s in self._dirty.values():
                s.clear()
        else:
            live = lambda s: [i for i in sorted(s) if i < cap and self._records[i] is not None]
            t = live(self._dirty["transform"])
            if t:
                self.ctx.set_local_matrices(np.stack([self._records[i].local_transform().matrix() for i in t]), np.array(t, np.uint32))
            fl = live(self._dirty["flags"])
            if fl:
                self.ctx.set_flags(np.array([self._records[i].flags_word() for i in fl], np.uint32), np.array(fl, np.uint32))
            m = live(self._dirty["mask"])
            if m:
                self.ctx.set_render_masks(np.array([self._records[i].render_mask for i in m], np.uint32), np.array(m, np.uint32))
            a = live(self._dirty["aabb"])
            if a:
                self.ctx.set_local_aabbs(np.stack([self._records[i].local_bounding_box for i in a]), np.array(a, np.uint32))
            for s in self._dirty.values():
                s.clear()
            self._upload_surfaces(reset=False)
        self._cache.clear()

    def _upload_surfaces(self, reset: bool):
        # surfaces are keyed by pool index, which a topology change does not move: the context rebuilds its
        # bone-slot tables itself (fyx_set_topology marks them dirty); only new surfaces are uploaded here
        for i, n in enumerate(self._records):
            if n is None:
                continue
            for s in n.surfaces:
                if s.surface_id is not None or not s.bones:
                    continue
                bones = np.array([b.index if self.is_valid_handle(b) else L.FYX_NONE for b in s.bones], np.uint32)
                ib = np.stack([self._records[b.index].inv_bind_pose_transform if self.is_valid_handle(b) else np.eye(4, dtype=f32).reshape(16) for b in s.bones])
                s.surface_id = self.ctx.add_skinned_surface(i, bones, ib, s.vertex_buffer, ANIMATED_VERTEX_LAYOUT)
                if s.skin_tangents and s.vertex_buffer is not None:  # before the blend shapes, which then lay out their tangent offsets
                    self.ctx.set_skinned_tangents(s.surface_id, s.vertex_buffer, 32, ANIMATED_VERTEX_LAYOUT.stride)
                self._surfaces_uploaded += 1
        self._upload_blend_shapes()

    def _upload_blend_shapes(self):
        """SurfaceData::blend_shapes_container -> fyx_set_blend_shapes once, Mesh::blend_shapes weights whenever they were touched."""
        for n in self._records:
            if n is None:
                continue
            for s in n.surfaces:
                c = s.blend_shapes_container
                if c is None or s.surface_id is None or c.blend_shape_storage is None:
                    continue
                w = np.array([b.weight for b in c.blend_shapes], np.float32)
                if not s._shapes_uploaded:
                    self.ctx.set_blend_shapes(s.surface_id, c.blend_shape_storage, w)
                    s._shapes_uploaded = True
                else:
                    self.ctx.set_blend_shape_weights(s.surface_id, w)

    def update(self, frame_size=None, dt: float = 1.0 / 60.0, switches=None):
        """Graph::update (graph/mod.rs:1459-1504) reduced to its hierarchical part: process_node_messages."""
        self._sync()
        self.ctx.update_transforms(L.UPDATE_INCREMENTAL)

    def update_hierarchical_data(self):
        """Graph::update_hierarchical_data (graph/mod.rs:1272-1292)."""
        self._sync()
        self.ctx.update_transforms(L.UPDATE_ALL)

    # ---- hierarchical queries (read back lazily, cached until the next change) ----
    def _fetch(self, key, fn):
        if key not in self._cache:
            self._cache[key] = fn()
        return self._cache[key]

    def _global_matrix(self, h: Handle) -> np.ndarray:
        return self._fetch("G", lambda: self.ctx.get_global_matrices())[h.index]

    def _global_flags(self, h: Handle) -> int:
        return int(self._fetch("F", lambda: self.ctx.get_global_flags())[h.index])

    def _world_aabb(self, h: Handle) -> np.ndarray:
        return self._fetch("A", lambda: self.ctx.get_world_aabbs())[h.index]

    def global_scale(self, h: Handle) -> np.ndarray:
        """Graph::global_scale (graph/mod.rs:1835-1845) — host-side product of local scales."""
        s = np.ones(3, f32)
        n = self.try_get_node(h)
        while n is not None:
            s = (s * n.local_transform().scale()).astype(f32)
            n = self.try_get_node(n.parent)
        return s


@dataclass
class ObserverPosition:
    """ObserverPosition (renderer/observer.rs:47-60)."""

    translation: np.ndarray
    z_near: float
    z_far: float
    view_matrix: np.ndarray
    projection_matrix: np.ndarray

    def view_projection_matrix(self) -> np.ndarray:
        return mat4_mul(self.projection_matrix, self.view_matrix)


def is_shadow_pass(render_pass_name: str) -> bool:
    """renderer::is_shadow_pass (renderer/mod.rs): the three shadow-map passes."""
    return render_pass_name in ("DirectionalShadow", "SpotShadow", "PointShadow")


class RenderDataBundleStorage:
    """The visible-node part of RenderDataBundleStorage (renderer/bundle.rs:873-1009)."""

    def __init__(self, handles: List[Handle], observer_position: ObserverPosition):
        self.visible_handles = handles
        self.observer_position = observer_position

    @staticmethod
    def from_graph(graph: Graph, render_mask: int, elapsed_time: float, observer_position: ObserverPosition,
                   render_pass_name: str = "GBuffer", options=None, dynamic_surface_cache=None) -> "RenderDataBundleStorage":
        return RenderDataBundleStorage.from_graph_multi(graph, [render_mask], [observer_position], [render_pass_name])[0]

    @staticmethod
    def from_graph_multi(graph: Graph, render_masks, observer_positions, render_pass_names) -> List["RenderDataBundleStorage"]:
        """Several observers in one pass over the node arrays (cube faces, CSM cascades)."""
        frusta = []
        for op in observer_positions:
            f = frustum_from_view_projection_matrix(op.view_projection_matrix())
            frusta.append(f if f is not None else frustum_default())  # unwrap_or_default, bundle.rs:893-896
        pass_flags = [L.PASS_SHADOW if is_shadow_pass(n) else 0 for n in render_pass_names]
        graph.ctx.cull(frusta, cam_mask=list(render_masks), pass_flags=pass_flags)
        out = []
        for i, op in enumerate(observer_positions):
            idx = graph.ctx.get_visible(i)
            out.append(RenderDataBundleStorage([Handle(int(k), graph._generation[int(k)]) for k in idx], op))
        return out
