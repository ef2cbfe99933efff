/*
 * fyrox_b200.h — C ABI of libfyrox_b200: Fyrox's per-frame render-prep hot path on B200 (sm_100a).
 *
 * The reference (Rust) has no FFI seam on this path (SURVEY.md §0 D6, §8b); these entry points are what
 * a Rust `-sys` shim would bind.  Each one names the reference interface it replaces (paths relative
 * to the Fyrox tree).  See INTEGRATION.md for the Rust-side binding and call sites.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes; no exceptions cross the boundary.
 *  - Return value: FYX_OK (0) or a negative fyx_status; fyx_last_error(ctx) gives a message.  This mirrors
 *    the reference's "log and continue" policy: invalid handles are skipped, never fatal
 *    (scene/graph/mod.rs:1167,1206; scene/mesh/mod.rs:785-791).
 *  - Node index i == Handle::index() of the node in Graph's Pool<Node>; capacity == Pool::get_capacity()
 *    (fyrox-core/src/pool/mod.rs:1104).  0xFFFFFFFF == Handle::NONE.
 *  - Matrices are 16 f32, column-major — nalgebra's Matrix4<f32> memory layout (bytemuck-castable).
 *    Only affine matrices (bottom row exactly 0,0,0,1) are accepted: that is all Transform::matrix()
 *    can produce (scene/transform.rs:476-539).
 *  - Caller owns every pointer it passes in; inputs are consumed before the call returns.  Pointers
 *    returned by fyx_get_visible* are library-owned and valid until the next fyx_cull*, fyx_render_prep or
 *    fyx_destroy on that context.
 *  - One fyx_ctx is used from one thread at a time (the engine's game-loop thread, engine/executor.rs:470-517).
 *  - There is no CPU fallback: every compute entry point runs hand-written sm_100a kernels and fails
 *    with FYX_ERR_CUDA if no device is usable.
 */
#ifndef FYROX_B200_H
#define FYROX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FYX_ABI_VERSION 2u
#define FYX_NONE 0xFFFFFFFFu
#define FYX_MAX_FRUSTA 8u      /* frusta per fyx_cull call: 1 camera, 3 CSM cascades, 6 cube faces (SURVEY §0 D5) */
#define FYX_MAX_BONES 255u     /* fyrox-material/src/shader/mod.rs:613; u8 indices scene/mesh/vertex.rs:154 */

typedef enum fyx_status {
    FYX_OK = 0,
    FYX_ERR_INVALID_ARGUMENT = -1,
    FYX_ERR_CUDA = -2,            /* CUDA runtime/driver error, or no sm_100 device */
    FYX_ERR_OUT_OF_MEMORY = -3,
    FYX_ERR_NOT_AFFINE = -4,      /* a matrix with a bottom row other than (0,0,0,1) or a non-finite entry */
    FYX_ERR_TOPOLOGY = -5,        /* cycle in parent[] / parent out of range */
    FYX_ERR_STATE = -6,           /* call order (e.g. cull before set_topology) */
    FYX_ERR_NCCL = -7,
    FYX_ERR_UNSUPPORTED = -8
} fyx_status;

/* Per-node flag word (inputs).  Bits 0..3 are Base's fields (scene/base.rs:412-432 and TrackedProperty
 * visibility/enabled :441-450), bit 4 the pool record's liveness, bit 5 "this node kind emits render
 * data and is frustum-tested" (Mesh::collect_render_data, scene/mesh/mod.rs:691-698). */
#define FYX_NODE_VISIBILITY      (1u << 0)
#define FYX_NODE_ENABLED         (1u << 1)
#define FYX_NODE_FRUSTUM_CULLING (1u << 2)
#define FYX_NODE_CAST_SHADOWS    (1u << 3)
#define FYX_NODE_ALIVE           (1u << 4)
#define FYX_NODE_RENDERABLE      (1u << 5)
#define FYX_NODE_LIGHT           (1u << 6)  /* the node is a BaseLight (point / spot / directional): fyx_cull_lights */
#define FYX_NODE_STATIC_BATCH    (1u << 7)  /* Mesh with BatchingMode::Static: when it is rendered for a frustum its children are
                                            * not visited for that frustum (RdcControlFlow::Break, scene/mesh/mod.rs:701-725) and its
                                            * instance carries the identity world matrix */
#define FYX_NODE_REFLECTION_PROBE (1u << 15) /* the node is a ReflectionProbe: fyx_select_reflection_probes */
#define FYX_NODE_INPUT_MASK      0x80FFu
/* Computed bits, readable through fyx_get_global_flags (Base::global_visibility / is_globally_enabled,
 * scene/base.rs:751-770) */
#define FYX_NODE_GLOBAL_VISIBILITY (1u << 8)
#define FYX_NODE_GLOBAL_ENABLED    (1u << 9)
#define FYX_NODE_REACHABLE         (1u << 10)  /* reached by the DFS from Graph::root (renderer/bundle.rs:1004) */

/* fyx_update_transforms flags */
#define FYX_UPDATE_INCREMENTAL 0u  /* Graph::update semantics: only sub-trees under changed nodes (process_node_messages) */
#define FYX_UPDATE_ALL         1u  /* Graph::update_hierarchical_data semantics: everything from the root */

/* fyx_cull pass flags */
#define FYX_PASS_SHADOW (1u << 0)  /* renderer::is_shadow_pass ⇒ nodes without cast_shadows are dropped */

typedef struct fyx_ctx fyx_ctx;

typedef struct fyx_config {
    uint32_t struct_size;   /* = sizeof(fyx_config) */
    int32_t  device;        /* CUDA device ordinal; -1 = current device */
    void    *stream;        /* cudaStream_t to launch on; NULL = the context creates its own */
    uint32_t flags;         /* reserved, 0 */
} fyx_config;

/* Frustum as fyrox-math/src/frustum.rs:26-30: planes 0 left,1 right,2 top,3 bottom,4 far,5 near, each
 * (nx,ny,nz,d) normalised; 8 corners in the order of frustum.rs:70-79. */
typedef struct fyx_frustum {
    float planes[6][4];
    float corners[8][3];
} fyx_frustum;

/* Where the attributes live inside one interleaved vertex (VertexBuffer layout, scene/mesh/buffer.rs:404-414).
 * AnimatedVertex (scene/mesh/vertex.rs:140-210): stride 68, position 0, normal 20, weights 48, indices 64. */
typedef struct fyx_vertex_layout {
    uint32_t stride;
    uint32_t position_offset;      /* f32 x3 */
    uint32_t normal_offset;        /* f32 x3 */
    uint32_t bone_weights_offset;  /* f32 x4 */
    uint32_t bone_indices_offset;  /* u8  x4 */
} fyx_vertex_layout;

/* Device-side durations of the stages run by the last fyx_render_prep / individual calls, in ms
 * (the GPU path's counterpart of GraphPerformanceStatistics, scene/graph/mod.rs:94-122).
 * Per-stage values are recorded by SYNCHRONOUS frames only: the events sit between the kernels of the frame's
 * programmatic-dependent-launch chain and would serialise it, so FYX_FRAME_ASYNC frames fill total_ms alone. */
typedef struct fyx_timings {
    float upload_ms;    /* H2D + scatter of changed local matrices / flags */
    float update_ms;    /* hierarchy + world AABB (+ fused cull) */
    float cull_ms;      /* stand-alone cull */
    float palette_ms;
    float skin_ms;
    float readback_ms;  /* D2H of visible counts + lists */
    float total_ms;
} fyx_timings;

/* ---- life cycle -------------------------------------------------------------------------- */
uint32_t    fyx_abi_version(void);
int32_t     fyx_create(const fyx_config *cfg, fyx_ctx **out_ctx);
void        fyx_destroy(fyx_ctx *ctx);
const char *fyx_last_error(const fyx_ctx *ctx);   /* ctx may be NULL: last error of fyx_create on this thread */
int32_t     fyx_sync(fyx_ctx *ctx);
/* Pinned host memory for zero-staging transfers (optional; any host pointer is accepted everywhere). */
void       *fyx_host_alloc(size_t bytes);
void        fyx_host_free(void *p);

/* ---- host-side math on the path (tiny, per frustum) ---------------------------------------- */
/* Frustum::from_view_projection_matrix (fyrox-math/src/frustum.rs:54-82) with Plane::from_abcd /
 * intersection_point (plane.rs:63-75,94-102).  Returns FYX_ERR_INVALID_ARGUMENT where the reference
 * returns None (a zero-length plane normal); callers then use fyx_frustum_default like
 * renderer/bundle.rs:893-896 (`unwrap_or_default`). */
int32_t fyx_frustum_from_view_projection_matrix(const float vp_m16[16], fyx_frustum *out);
void    fyx_frustum_default(fyx_frustum *out);                      /* frustum.rs:32-43 */
/* Matrix4 * Matrix4 in nalgebra's accumulation order (projection * view, renderer/bundle.rs:894). */
void    fyx_mat4_mul(const float a_m16[16], const float b_m16[16], float out_m16[16]);

/* ---- scene description (on load / when the hierarchy changes) ------------------------------ */
/* Replaces the pointer graph walked by Graph::update_hierarchical_data (scene/graph/mod.rs:1272-1292):
 * parent[i] = Base::parent index or FYX_NONE; flags[i] = FYX_NODE_* input bits; render_mask[i] =
 * Base::render_mask (NULL = all ones); local_aabb_minmax = 6 f32 per node (min xyz, max xyz) —
 * NodeTrait::local_bounding_box (Mesh: scene/mesh/mod.rs:631-656; others the unit box, scene/base.rs:733-735;
 * NULL = unit box everywhere).  root = Graph::root index.  global_index (optional, NULL = identity) is the
 * value written to visible lists for node i — used when a context holds one shard of a larger graph.
 * Marks every node changed (like Base::on_connected_to_graph, scene/base.rs:520-540): the next update recomputes
 * every global matrix and world box.
 * What the call keeps: everything that is per node but not an argument here — local matrices, TRS records, transform
 * statics, bundle ids, LOD ranges, skinned surfaces and animations — stays with its node index (the data moves to the
 * node's new place on the device); a node index that was not alive before the call starts from the defaults (identity
 * local matrix ...).  The DFS order is kept while `capacity` is unchanged.  So the add / link / remove sequence of
 * INTEGRATION.md is: fyx_set_topology with the new columns, then upload the matrices of the NEW or changed nodes only. */
int32_t fyx_set_topology(fyx_ctx *ctx, uint32_t capacity, uint32_t root, const uint32_t *parent,
                         const uint32_t *flags, const uint32_t *render_mask, const float *local_aabb_minmax,
                         const uint32_t *global_index);

/* Optional.  preorder_rank[i] = position of node i in the pre-order DFS from the root in `children` order — the
 * order Graph::update_global_transform_recursively visits nodes (scene/graph/mod.rs:1199-1241).  Only one thing
 * depends on it: Mesh::on_global_transform_changed (scene/mesh/mod.rs:676-682) folds each bone's position AS STORED
 * when the mesh is visited, so a bone that comes later in that order contributes its position from before the
 * update.  With the order given, such bones are snapshotted before every update and the skinned-mesh boxes equal
 * the reference's; without it (or NULL) every bone contributes its new position — identical whenever skeletons
 * precede their meshes.  Kept by fyx_set_topology while the capacity is unchanged. */
int32_t fyx_set_dfs_order(fyx_ctx *ctx, uint32_t capacity, const uint32_t *preorder_rank);

/* Transform::matrix() of `count` nodes (scene/transform.rs:544-550); idx NULL = nodes 0..count-1.
 * Equivalent of `local_transform_mut()` → NodeMessageKind::TransformChanged (scene/base.rs:343-352). */
int32_t fyx_set_local_matrices(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const float *m16_colmajor);
/* The same, but the library evaluates Transform::calculate_local_transform (scene/transform.rs:421-540) on the
 * device from the Transform's fields instead of receiving the 64-byte matrix: 40 B per changed node go over
 * PCIe instead of 64.  position / rotation (unit quaternion i,j,k,w) / scale are what animation writes every
 * frame (AnimationPose::apply, scene/animation/mod.rs:147-179); the remaining fields of Transform rarely
 * change and are set once with fyx_set_transform_statics (default: identity pre-rotation and post-rotation
 * matrix, zero pivots/offsets — TransformBuilder's defaults, scene/transform.rs:176-200). */
typedef struct fyx_trs {
    float position[3];
    float rotation[4];
    float scale[3];
} fyx_trs;
typedef struct fyx_transform_statics {
    float pre_rotation[4];            /* unit quaternion i,j,k,w */
    float post_rotation_matrix[9];    /* column-major 3x3: Transform::post_rotation_matrix (inverse of the post rotation, :160-172) */
    float rotation_offset[3], rotation_pivot[3], scaling_offset[3], scaling_pivot[3];
} fyx_transform_statics;
int32_t fyx_set_local_trs(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const fyx_trs *trs);
/* Transform::set_rotation only (what skeletal animation does to most bones every frame): 16 B per node; position and
 * scale stay what the node's last fyx_set_local_trs sent (identity for a node that never got one). */
int32_t fyx_set_local_rotations(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const float *quat_ijkw);
int32_t fyx_set_transform_statics(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const fyx_transform_statics *statics);
/* Base::set_visibility / set_enabled / frustum_culling / cast_shadows (VisibilityChanged / EnabledFlagChanged). */
int32_t fyx_set_flags(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const uint32_t *flags);
int32_t fyx_set_render_masks(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const uint32_t *render_mask);
int32_t fyx_set_local_aabbs(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const float *aabb_minmax);

/* One skinned Surface of Mesh node `mesh_node` (scene/mesh/surface.rs:1249-1271): `bone_nodes` = Surface::bones
 * indices (≤255), inv_bind_m16 = each bone's Base::inv_bind_pose_transform (scene/base.rs:482), verts = the
 * surface's VertexBuffer bytes (n_verts * layout->stride).  Surfaces of one mesh are folded into its world
 * AABB in call order (scene/mesh/mod.rs:676-682).  verts may be NULL with n_verts 0 (palette only). */
int32_t fyx_add_skinned_surface(fyx_ctx *ctx, uint32_t mesh_node, uint32_t n_bones, const uint32_t *bone_nodes,
                                const float *inv_bind_m16, uint32_t n_verts, const void *verts,
                                const fyx_vertex_layout *layout, uint32_t *out_surface_id);
/* Optional: size the device-side bone / vertex tables once for `total_bones` palette entries and
 * `total_verts` vertices (sum over all surfaces to be added) instead of growing them on demand. */
int32_t fyx_reserve_skinning(fyx_ctx *ctx, uint64_t total_bones, uint64_t total_verts);
/* Finish a batch of fyx_add_skinned_surface calls (builds the device-side bone/vertex tables). Called
 * implicitly by the first per-frame call that needs them. */
int32_t fyx_commit_surfaces(fyx_ctx *ctx);

/* ---- per frame ----------------------------------------------------------------------------- */
/* Graph::update → process_node_messages (scene/graph/mod.rs:1303-1399, 1459-1473): global transforms
 * (update_global_transform_recursively :1199-1241), global visibility / enabled (:1166-1197), world AABBs
 * (AxisAlignedBoundingBox::transform, fyrox-math/src/aabb.rs:264-287; Mesh::on_global_transform_changed,
 * scene/mesh/mod.rs:667-689). */
int32_t fyx_update_transforms(fyx_ctx *ctx, uint32_t update_flags);

/* RenderDataBundleStorage::from_graph reduced to its visible-node set (renderer/bundle.rs:873-1009):
 * for each frustum f, the nodes for which NodeTrait::should_be_rendered(frustum, cam_mask[f])
 * (scene/node/mod.rs:231-256, Frustum::is_intersects_aabb fyrox-math/src/frustum.rs:222-245) holds, that are
 * alive, renderable and reachable from the root, and (pass_flags[f] & FYX_PASS_SHADOW) ⇒ cast_shadows.
 * cam_mask NULL = all ones; pass_flags NULL = 0.  The list is a SET: its order is unspecified. */
int32_t fyx_cull(fyx_ctx *ctx, uint32_t n_frusta, const fyx_frustum *frusta, const uint32_t *cam_mask,
                 const uint32_t *pass_flags);
/* fyx_update_transforms + fyx_cull in one pass over the node arrays (world AABBs stay in registers). */
int32_t fyx_update_and_cull(fyx_ctx *ctx, uint32_t update_flags, uint32_t n_frusta, const fyx_frustum *frusta,
                            const uint32_t *cam_mask, const uint32_t *pass_flags);
/* Visible list of frustum f as node indices (global_index values): host copy (pinned) ... */
int32_t fyx_get_visible(fyx_ctx *ctx, uint32_t frustum, const uint32_t **out_idx, uint32_t *out_count);
/* ... or device-resident (for a GPU consumer / a collective); *d_count points at one device u32. */
int32_t fyx_get_visible_device(fyx_ctx *ctx, uint32_t frustum, const uint32_t **d_idx, const uint32_t **d_count);

/* N4 (light list) — the `collect_lights` part of RenderDataBundleStorage::from_graph (renderer/bundle.rs:926-974): for
 * every frustum of the most recent cull, the FYX_NODE_LIGHT nodes whose world bounding box the frustum intersects and
 * that are globally visible and enabled (no reachability / render-mask / frustum_culling-flag test, as in the
 * reference).  Lists come back in ascending node index = the reference's pool order.  Lights in sub-trees detached from
 * the root are outside the contract: the reference never updates such sub-trees, this library updates every tree. */
int32_t fyx_cull_lights(fyx_ctx *ctx);
/* The reflection-probe part of the same loop (renderer/bundle.rs:918-925): per observer of fyx_set_observers the LAST node in pool
 * order that carries FYX_NODE_REFLECTION_PROBE and whose world bounding box contains the observer's translation (inclusive) —
 * `storage.environment_map`; FYX_NONE = none.  out_probe receives one node index per observer. */
int32_t fyx_select_reflection_probes(fyx_ctx *ctx, uint32_t count, uint32_t *out_probe);
int32_t fyx_get_visible_lights(fyx_ctx *ctx, uint32_t frustum, const uint32_t **out_idx, uint32_t *out_count);

/* N4 (LOD filter) — the lod_filter of RenderDataBundleStorage::from_graph (renderer/bundle.rs:898-916, 988-1004): a node
 * that is an object of a LOD level is visible for an observer only while its normalised distance
 * (|observer.translation − global_position| − z_near) / (z_far − z_near) lies in the level's [begin, end]; a node that is
 * filtered out hides its whole sub-tree (the DFS does not descend).
 * fyx_set_lod_ranges: per LOD object the range of the level it belongs to (2 floats each: begin, end; begin = NaN removes
 * the node from LOD control).  The host resolves "listed in several levels" the way the reference's loop does — owners in
 * pool order, levels and objects in order, the last write wins.  Carried over by fyx_set_topology with the node indices.
 * fyx_set_observers: ObserverPosition::{translation, z_near, z_far} of the frusta of the culls that follow, one per
 * frustum (count 0 = no LOD filtering).  While both are set the cull runs un-fused: update, then one small pass per
 * hierarchy level that propagates the filter bits from parents to children, then the cull over all nodes. */
typedef struct fyx_observer {
    float translation[3];
    float z_near, z_far;
} fyx_observer;
int32_t fyx_set_lod_ranges(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const float *begin_end);
int32_t fyx_set_observers(fyx_ctx *ctx, uint32_t count, const fyx_observer *observers);

/* ---- N4: blend shapes (morph targets) ahead of the skinning ------------------------------------------------ */
/* The standard shader adds, for every blend shape i of the surface in order, offsets.position * weight to the vertex
 * position and offsets.normal * weight to the normal BEFORE skinning (fyrox-material/src/shader/standard/opengl/
 * standard.shader:167-173), weight = BlendShape::weight / 100 (scene/mesh/mod.rs:794-798).  `records` is the content of
 * BlendShapesContainer::blend_shape_storage as from_lists builds it (scene/mesh/surface.rs:92-218): n_shapes layers of
 * layer_stride (= width * height >= n_verts) records of 9 binary16 values — position, normal, tangent offsets of vertex
 * v at record v of the layer.  The tangent offsets are laid out only for a surface that has skinned tangents at the time of
 * the call (fyx_set_skinned_tangents, which must come first); other surfaces ignore them.  `weights` = the
 * BlendShape::weight values (0..100), NULL = 100 each (BlendShape::default()).  n_shapes = 0 removes them.
 * Costs 12 more bytes read per vertex and shape in fyx_skin (18 on a tangent surface); surfaces without shapes are unaffected. */
#define FYX_MAX_BLEND_SHAPES 128u /* ShaderDefinition::MAX_BLEND_SHAPE_WEIGHT_GROUPS * 4, fyrox-material/src/shader/mod.rs:616 */
int32_t fyx_set_blend_shapes(fyx_ctx *ctx, uint32_t surface_id, uint32_t n_shapes, const void *records, uint32_t layer_stride,
                             const float *weights);
int32_t fyx_set_blend_shape_weights(fyx_ctx *ctx, uint32_t surface_id, uint32_t n, const float *weights);

/* ---- skinned tangents (opt-in, per surface) ------------------------------------------------------------------ */
/* The standard shader skins the tangent as it skins the normal (standard.shader:197-200): acc += (mat3(P[idx_k]) * t) * w_k,
 * after the blend shapes added offsets.tangent * weight (:167-173).  A normal-mapped renderer needs the skinned tangent for
 * its binormal, w * cross(normal, tangent).  fyx_set_skinned_tangents adds a third skinned stream to one surface: `verts`
 * = the surface's VertexBuffer bytes again (n_verts records of `stride` bytes) with the tangent as f32 x4 at tangent_offset
 * (32 in AnimatedVertex); only .xyz is skinned, .w (the handedness) stays in the renderer's own vertex buffer.  Normalising,
 * the world matrix and the binormal stay with the renderer, as for normals.  verts = NULL turns the surface's tangents off.
 * FYX_ERR_INVALID_ARGUMENT: stride or tangent_offset not a multiple of 4, or tangent_offset + 16 > stride.
 * FYX_ERR_STATE: the surface already has blend shapes (call this before fyx_set_blend_shapes).  Surfaces without tangents
 * run exactly as before; the tangent data belongs to the surface and survives fyx_set_topology.  Costs 12 bytes read and
 * 12 written per vertex of a tangent surface in fyx_skin. */
int32_t fyx_set_skinned_tangents(fyx_ctx *ctx, uint32_t surface_id, const void *verts, uint32_t stride, uint32_t tangent_offset);
/* The skinned tangents of the last fyx_skin / render prep, packed xyz (n_verts*3); FYX_ERR_STATE for a surface without tangents. */
int32_t fyx_get_skinned_tangents(fyx_ctx *ctx, uint32_t surface_id, float *out_tan3);
int32_t fyx_get_skinned_tangents_device(fyx_ctx *ctx, uint32_t surface_id, const float **d_tan3);

/* SurfaceInstanceData::bone_matrices for every skinned surface (scene/mesh/mod.rs:781-793):
 * P[k] = bone_k.global_transform * bone_k.inv_bind_pose_transform; dead / FYX_NONE bone ⇒ identity. */
int32_t fyx_build_palettes(fyx_ctx *ctx);
/* Linear-blend skinning of every skinned surface: positions as Mesh::accurate_world_bounding_box
 * (scene/mesh/mod.rs:501-522), normals as the standard shader (fyrox-material/src/shader/standard/opengl/
 * standard.shader:192-195) — into device-resident position / normal streams; and the tangents of the surfaces that have
 * them (fyx_set_skinned_tangents, standard.shader:197-200) into a third stream. */
int32_t fyx_skin(fyx_ctx *ctx);

/* One whole frame of render prep, in stream order, with one host synchronisation at the end:
 * upload changed local matrices → update (+cull) → palettes → skin → visible lists to the host.
 * Any of the parts may be empty (count 0 / n_frusta 0 / no surfaces). */
typedef struct fyx_frame_desc {
    uint32_t struct_size;
    uint32_t update_flags;
    uint32_t n_changed;            /* changed local matrices this frame */
    const uint32_t *changed_idx;   /* NULL = nodes 0..n_changed-1 */
    const float *changed_m16;      /* n_changed * 16 f32 ... */
    const fyx_trs *changed_trs;    /* ... or, if non-NULL, n_changed fyx_trs records (changed_m16 ignored) */
    const float *changed_rot;      /* ... or, if non-NULL, n_changed rotations (4 f32 each; the others ignored) */
    uint32_t n_frusta;
    const fyx_frustum *frusta;
    const uint32_t *cam_mask;
    const uint32_t *pass_flags;
    uint32_t do_palettes;
    uint32_t do_skin;
    uint32_t readback_visible;     /* copy counts + lists to the host before returning */
    uint32_t flags;                /* FYX_FRAME_* */
    /* since ABI 2 (struct_size tells which fields the caller has): */
    uint32_t do_animate;           /* first run fyx_animate(animate_dt): AnimationPlayer::update before Graph::update */
    float animate_dt;
} fyx_frame_desc;
/* Do not synchronise with the host at the end of fyx_render_prep: the frame is only enqueued.  Inputs must
 * stay untouched until the frame is waited for (fyx_frame_wait / fyx_sync).  Pinned inputs are uploaded on
 * a copy stream into alternating staging buffers, so the upload of frame i+1 overlaps the kernels of
 * frame i.  With readback_visible the read-back is deferred: at most two such frames may be in flight,
 * fyx_frame_wait collects the oldest one and makes its visible lists the ones fyx_get_visible returns. */
#define FYX_FRAME_ASYNC (1u << 0)
/* Multi-GPU (after fyx_comm_init): all-gather the frame's visible lists as soon as the cull is done, on a
 * separate stream, overlapped with the palette / skinning kernels of the same frame; the frame is complete
 * when the gathered lists are (fyx_get_visible_gathered*).  Collective: every rank issues the frame.
 * With readback_visible every rank also copies its OWN lists into the node-wide host segment (one PCIe link per rank);
 * fyx_get_visible_gathered on any rank then returns the whole lists from that segment and fyx_get_visible the rank's
 * own part of it (fyx_comm_mode tells whether the segment is in use; without it the host copy comes from the rank's
 * device). */
#define FYX_FRAME_ALLGATHER (1u << 1)
/* With FYX_FRAME_ALLGATHER on a pipelined (async + read-back) frame and NO host segment (FYX_HOSTSEG=0 or not available):
 * bring only THIS rank's lists to the host (fyx_get_visible); the gathered lists stay device-resident.  One process of the
 * job — the one that feeds the CPU-side renderer — leaves it off and receives the whole lists through its pinned copy; the
 * others do not multiply that PCIe traffic by the number of GPUs.  With the host segment the flag changes nothing: every
 * rank copies its own lists only. */
#define FYX_FRAME_READBACK_OWN (1u << 2)
int32_t fyx_frame_wait(fyx_ctx *ctx);
int32_t fyx_render_prep(fyx_ctx *ctx, const fyx_frame_desc *frame);

/* ---- read-back (tests, tools, and the parts of the engine that stay on the CPU) -------------- */
int32_t fyx_get_global_matrices(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, float *out_m16);   /* Base::global_transform */
int32_t fyx_get_world_aabbs(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, float *out_minmax);    /* NodeTrait::world_bounding_box */
int32_t fyx_get_global_flags(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, uint32_t *out_flags);
int32_t fyx_get_palette(fyx_ctx *ctx, uint32_t surface_id, float *out_m16 /* n_bones*16 */);
int32_t fyx_get_skinned(fyx_ctx *ctx, uint32_t surface_id, float *out_pos3, float *out_nrm3 /* n_verts*3 each; either may be NULL */);
int32_t fyx_get_skinned_device(fyx_ctx *ctx, uint32_t surface_id, const float **d_pos3, const float **d_nrm3);
int32_t fyx_get_timings(fyx_ctx *ctx, fyx_timings *out);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t fyx_kernel_launch_count(const fyx_ctx *ctx);

/* ---- N2: animation sampling on the device (SURVEY §8f) ---------------------------------------- */
/* What AnimationPlayer nodes do on the CPU before Graph::update (scene/animation/mod.rs:83-88,340-346): every
 * enabled animation ticks — its tracks' curves are sampled at the current time position (fyrox-animation/src/
 * lib.rs:895-914, container.rs:162-301, fyrox-math/src/curve.rs:252-309), the pose is applied to the target
 * nodes' position / rotation / scale (scene/animation/mod.rs:147-179) and the time position advances
 * (lib.rs:471-496, 432-440).  With the curves resident in HBM nothing is uploaded per frame.
 * Properties no track writes keep the value of the node's last fyx_set_local_trs record (identity if none);
 * pivots / offsets / pre- and post-rotation come from fyx_set_transform_statics.
 * Parity: Vector3 and UnitQuaternion tracks bit-exact; UnitQuaternionEuler tracks use sin/cos (platform libm in the
 * reference): ~1e-7 absolute on the quaternion.  Signals, root motion, property bindings and the blend-machine
 * (ABSM) layers are not modelled. */
#define FYX_KEY_CONSTANT 0u /* CurveKeyKind (fyrox-math/src/curve.rs:33-45) */
#define FYX_KEY_LINEAR 1u
#define FYX_KEY_CUBIC 2u
typedef struct fyx_curve_key {
    float location, value;
    uint32_t kind;                     /* FYX_KEY_* */
    float left_tangent, right_tangent; /* tan(angle), Cubic only */
} fyx_curve_key;

#define FYX_TV_REAL 0u /* TrackValueKind (fyrox-animation/src/container.rs:41-54) */
#define FYX_TV_VECTOR2 1u
#define FYX_TV_VECTOR3 2u
#define FYX_TV_VECTOR4 3u
#define FYX_TV_QUAT_EULER 4u
#define FYX_TV_QUAT 5u
#define FYX_BIND_POSITION 0u /* ValueBinding (fyrox-animation/src/value.rs:358-374) */
#define FYX_BIND_SCALE 1u
#define FYX_BIND_ROTATION 2u
typedef struct fyx_anim_track {
    uint32_t target_node;  /* TrackBinding::target (node index) */
    uint32_t binding;      /* FYX_BIND_* */
    uint32_t value_kind;   /* FYX_TV_* */
    uint32_t enabled;      /* TrackBinding::enabled */
    uint32_t n_curves;     /* TrackDataContainer::curves.len(): fewer than the kind needs = fetch returns None */
    uint32_t first_key[4]; /* curve c = keys[first_key[c] .. first_key[c] + n_keys[c]), sorted by location */
    uint32_t n_keys[4];
} fyx_anim_track;

typedef struct fyx_animation_desc {
    uint32_t struct_size;
    uint32_t n_tracks;
    const fyx_anim_track *tracks; /* in AnimationTracksData::tracks order */
    uint32_t n_keys;
    const fyx_curve_key *keys;
    float speed;                  /* Animation defaults (lib.rs:922-945): 1.0 */
    float time_position;
    float time_slice_start, time_slice_end;
    uint32_t looped;
    uint32_t enabled;
} fyx_animation_desc;

/* Add an animation; ids are 0,1,2,... in call order = the order update_animations walks them. */
int32_t fyx_anim_add(fyx_ctx *ctx, const fyx_animation_desc *desc, uint32_t *out_id);
int32_t fyx_anim_clear(fyx_ctx *ctx);
int32_t fyx_anim_set_enabled(fyx_ctx *ctx, uint32_t anim, uint32_t enabled);                        /* Animation::set_enabled */
int32_t fyx_anim_set_track_enabled(fyx_ctx *ctx, uint32_t anim, uint32_t track, uint32_t enabled);  /* TrackBinding::set_enabled */
int32_t fyx_anim_set_speed(fyx_ctx *ctx, uint32_t anim, float speed);
int32_t fyx_anim_set_time_position(fyx_ctx *ctx, uint32_t anim, float time); /* wraps / clamps into the time slice (lib.rs:432-440) */
int32_t fyx_anim_get_time_positions(fyx_ctx *ctx, uint32_t first, uint32_t count, float *out);
/* Pose blending, the smallest useful subset of the blend machine (fyrox-animation/src/machine): the listed animations
 * stop being applied directly (AnimationPlayer::auto_apply = false) and become, in this order, the PlayAnimation sources
 * of ONE PoseNode::BlendAnimations with constant weights (machine/node/blend.rs:136-166) in a one-layer, one-state
 * machine: every enabled source still ticks (machine/mod.rs:366-372; a disabled one keeps contributing the pose of its
 * last tick), the output pose takes a clone of the first source that has values for a node and blends every later
 * source into it per binding — AnimationPose::blend_with / TrackValue::blend_with (pose.rs:41-101, value.rs:201-227:
 * nalgebra lerp for vectors, shortest-way nlerp for rotations) — and is then applied.  Groups are applied after the
 * directly applied animations, in creation order.  Restrictions: Vector3 / UnitQuaternion(Euler) tracks only, one track
 * per (node, property) and animation, an animation in at most one group.  Transitions, parameters, masks, blend
 * spaces, layers > 1: not modelled. */
int32_t fyx_anim_blend_group(fyx_ctx *ctx, uint32_t n, const uint32_t *anims, const float *weights, uint32_t *out_group);
int32_t fyx_anim_set_blend_weights(fyx_ctx *ctx, uint32_t group, uint32_t n, const float *weights);
/* AnimationContainer::update_animations(dt) for every animation of the context.  The touched nodes are marked
 * changed exactly like fyx_set_local_trs; follow with fyx_update_transforms / fyx_render_prep. */
int32_t fyx_animate(fyx_ctx *ctx, float dt);

/* ---- N3: draw-prep after the cull (SURVEY §8f) ------------------------------------------------ */
/* What RenderDataBundleStorage::push and RenderDataBundle::write_uniforms do per visible surface on the CPU
 * (renderer/bundle.rs:1248-1278, 483-487), for nodes with ONE surface: the instances of a frustum's visible
 * list grouped by bundle, each with its sort index, world matrix and view_projection * world. */

/* Meshes with several surfaces (Mesh::surfaces): Mesh::collect_render_data pushes ONE SurfaceInstanceData per surface, each
 * into the bundle of ITS (material, surface data, render path) key and with ITS bones, all with the node's sort index; the
 * world matrix is the identity for a skinned surface and the node's global transform otherwise (scene/mesh/mod.rs:726-805).
 * For node idx[i] the surfaces are entries [first[i], first[i+1]) of bundle_ids / skin_surface (first has count + 1 entries):
 * bundle_ids[k] = the dense bundle id of surface k, skin_surface[k] = the fyx surface id (fyx_add_skinned_surface) whose
 * palette skins it, FYX_NONE (or skin_surface == NULL) = unskinned.  Nodes never listed keep the default: one surface in the
 * node's bundle id (fyx_set_bundle_ids), skinned iff the node has a skinned surface.  A count of 0 surfaces restores the default. */
int32_t fyx_set_node_surfaces(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const uint32_t *first, const uint32_t *bundle_ids,
                              const uint32_t *skin_surface);
/* Per-node bundle id = the host's dense id for the (material, surface data, render path) key that push()
 * hashes (renderer/bundle.rs:1253-1257); every node starts in bundle 0.  idx NULL = nodes 0..count-1. */
int32_t fyx_set_bundle_ids(fyx_ctx *ctx, uint32_t count, const uint32_t *idx, const uint32_t *bundle_ids);
/* Ask the culls that follow to also record where each visible node lives in HBM (4 more bytes written per
 * visible entry); required before fyx_pack_instances. */
int32_t fyx_enable_instances(fyx_ctx *ctx, uint32_t enable);

typedef struct fyx_bundle {
    uint32_t id;          /* the bundle id given to fyx_set_bundle_ids */
    uint32_t first;       /* first instance of the bundle in the packed arrays */
    uint32_t count;       /* RenderDataBundle::instances.len() */
    uint32_t reserved;
    uint64_t sort_index;  /* RenderDataBundle::sort_index: that of the instance pushed first (bundle.rs:1264-1268), i.e.
                           * first in the DFS order given to fyx_set_dfs_order, else the lowest node index */
} fyx_bundle;

typedef struct fyx_instances {
    uint32_t count;             /* instances: one per (visible node, surface) */
    uint32_t n_bundles;         /* non-empty bundles */
    const uint32_t *node;       /* [count]   SurfaceInstanceData::node_handle (index) */
    const uint64_t *sort_index; /* [count]   RenderContext::calculate_sorting_index(global_position) (bundle.rs:118-127) */
    const float *matrices;      /* [count*32] per instance: world_transform (identity for a skinned surface,
                                 * scene/mesh/mod.rs:733-737), then view_projection * world_transform (bundle.rs:485);
                                 * both column-major — the first 128 bytes of the instance uniform block */
    const fyx_bundle *bundles;  /* [n_bundles] ascending id; bundle b owns instances [first, first+count) in unspecified order */
} fyx_instances;

/* Pack the visible list of `frustum` (of the most recent cull, made with instances enabled) for an observer
 * with the given view and view-projection matrices (ObserverPosition, renderer/observer.rs). */
int32_t fyx_pack_instances(fyx_ctx *ctx, uint32_t frustum, const float *view_m16, const float *view_projection_m16);
/* [count] ordinal of each packed instance's surface within its node (host copy; 0 everywhere without fyx_set_node_surfaces). */
int32_t fyx_get_instance_surfaces(fyx_ctx *ctx, uint32_t frustum, const uint32_t **out_ordinal);
/* Result of the last fyx_pack_instances for that frustum: pointers to pinned host copies ... */
int32_t fyx_get_instances(fyx_ctx *ctx, uint32_t frustum, fyx_instances *out);
/* ... or to the device-resident arrays (count / n_bundles still come back as host values). */
int32_t fyx_get_instances_device(fyx_ctx *ctx, uint32_t frustum, fyx_instances *out);

/* Bone matrices of the packed instances, as RenderDataBundle::write_uniforms lays them out (renderer/bundle.rs:484-496):
 * every instance whose node has a skinned surface gets a block of FYX_MAX_BONES (255 = ShaderDefinition::
 * MAX_BONE_MATRICES) column-major mat4 — its SurfaceInstanceData::bone_matrices, then all-zero matrices — and an
 * unskinned instance gets none (bone_matrices_block = None).  Uses the palettes of the last fyx_build_palettes /
 * fyx_render_prep; call after fyx_pack_instances.  The surface that skins an instance is the one named by
 * fyx_set_node_surfaces, else the node's first skinned surface. */
typedef struct fyx_bone_blocks {
    uint32_t count;                    /* instances == fyx_instances.count */
    uint32_t n_blocks;                 /* skinned instances */
    const uint32_t *block_of_instance; /* [count] block of packed instance i, FYX_NONE = unskinned          (device memory) */
    const float *blocks;               /* [n_blocks * 255 * 16], 16 320 bytes per block, in unspecified order (device memory) */
} fyx_bone_blocks;
int32_t fyx_pack_bone_matrices(fyx_ctx *ctx, uint32_t frustum);
int32_t fyx_get_bone_matrix_blocks_device(fyx_ctx *ctx, uint32_t frustum, fyx_bone_blocks *out);
/* Host copy of one instance's block (out_255x16 may be NULL to ask only whether it has one). */
int32_t fyx_get_bone_matrix_block(fyx_ctx *ctx, uint32_t frustum, uint32_t instance, float *out_255x16, uint32_t *out_has_block);

/* ---- multi-GPU: one context per GPU, one process per GPU ------------------------------------- */
/* The node array is sharded (sub-trees + replicated ancestors, SURVEY §8e); each context culls its
 * shard; the per-frustum visible lists are all-gathered with NCCL over NVLink so every rank holds
 * the whole list.  Rank 0 obtains an id, the host broadcasts it, every rank calls fyx_comm_init. */
#define FYX_COMM_ID_BYTES 128
int32_t fyx_comm_get_unique_id(void *out_id128);
/* Collective.  The exchange buffers are built at the first gathered frame that follows (also collective: every rank
 * issues gathered frames in lockstep) and sized for every rank's node count at that time; call fyx_comm_init again on
 * every rank after a topology change that grows a shard. */
int32_t fyx_comm_init(fyx_ctx *ctx, int32_t nranks, int32_t rank, const void *id128);
/* How this context exchanges the lists (bit set), decided collectively at the first gathered frame:
 *   FYX_COMM_NCCL          NCCL is initialised (always; it is also the bootstrap channel of the other two)
 *   FYX_COMM_PEER_STORES   the device-side all-gather is done by direct stores into the peers' cudaIpc-mapped list
 *                          buffers over NVLink (no host synchronisation, no padded slots); otherwise ncclAllGather
 *   FYX_COMM_HOST_SEGMENT  the host copy of the gathered lists is assembled in one node-wide host segment: every rank
 *                          DMA-copies its own lists there over its own PCIe link
 *   FYX_COMM_UNDECIDED     no gathered frame has run yet
 * Environment (read by fyx_comm_init): FYX_EXCHANGE=nccl keeps the collective on NCCL, FYX_HOSTSEG=0 keeps private
 * host copies. */
#define FYX_COMM_NCCL 1u
#define FYX_COMM_PEER_STORES 2u
#define FYX_COMM_HOST_SEGMENT 4u
#define FYX_COMM_UNDECIDED 8u
uint32_t fyx_comm_mode(const fyx_ctx *ctx);
/* The most recent COMPLETED exchange of this rank, timed with CUDA events on the collective stream (waits for it). */
typedef struct fyx_comm_stats {
    uint64_t epoch;          /* number of the gathered frame */
    uint64_t entries_own;    /* visible entries this rank contributed (all frusta) */
    uint64_t entries_total;  /* entries of the gathered lists (all frusta) */
    uint64_t egress_bytes;   /* bytes this rank stored into OTHER ranks' memory: 4 * entries_own * (nranks - 1) (peer form) */
    float device_ms;         /* from the first kernel / collective of the exchange to its last one, incl. waiting for peers */
    uint32_t mode;           /* fyx_comm_mode at that time */
} fyx_comm_stats;
int32_t fyx_comm_get_stats(fyx_ctx *ctx, fyx_comm_stats *out);
/* All-gather the visible lists of the last cull.  Collective: every rank calls it for the same frame. */
int32_t fyx_allgather_visible(fyx_ctx *ctx);
/* Gathered list of frustum f: concatenation over ranks (device-resident and, if readback, on the host). */
int32_t fyx_get_visible_gathered(fyx_ctx *ctx, uint32_t frustum, const uint32_t **out_idx, uint32_t *out_count);
int32_t fyx_get_visible_gathered_device(fyx_ctx *ctx, uint32_t frustum, const uint32_t **d_idx, uint32_t *out_count);

#ifdef __cplusplus
}
#endif
#endif /* FYROX_B200_H */
