// fyx_internal.h — device data layout and kernel launchers shared by fyx_api.cu / fyx_kernels.cu.
//
// HBM layout (DESIGN.md §3).  Nodes live in SLOT order = sorted by (depth, node index), so every
// hierarchy level is one contiguous, coalesced range and a parent is always in an earlier range.
// All per-node columns are SoA planes indexed by slot:
//   L[3], G[3]   float4 rows of the affine local / global matrix (48 B each; bottom row implicit)
//   la[3], wa[3] float2 (min_i,max_i) pairs of the local / world AABB (24 B each)
//   parent       u32 parent slot (FYX_NONE = none)      flags  u32 (input bits + computed bits)
//   mask         u32 Base::render_mask                  gidx   u32 node index emitted to visible lists
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/fyrox_b200.h"
#include "fyx_math.cuh"

namespace fyx {

// internal flag bits (above the public ones)
constexpr uint32_t F_DIRTY_SELF = 1u << 11; // local matrix / topology changed since the last update
constexpr uint32_t F_DIRTY = 1u << 12;      // in a changed sub-tree during the last update
constexpr uint32_t F_SKINNED = 1u << 13;    // Mesh with at least one skinned surface
constexpr uint32_t F_ROOT = 1u << 14;       // Graph::root

constexpr int kCountStride = 32; // u32s between per-frustum counters (128 B: one L2 line each)
constexpr int kBlock = 256;

struct NodeArrays {
    uint32_t cap; // number of slots (alive nodes)
    uint32_t *parent;
    uint32_t *flags;
    uint32_t *mask;
    uint32_t *gidx;
    uint8_t *vis; // per slot: bit f = visible in frustum f of the current cull (deferred compaction, k_compact_vis)
    float4 *L[3];
    float4 *G[3];
    float2 *la[3];
    float2 *wa[3];
};

struct CullParams {
    int nf;
    FrustumDev f[FYX_MAX_FRUSTA];
    uint32_t *out[FYX_MAX_FRUSTA]; // visible lists
    uint32_t *out_slot[FYX_MAX_FRUSTA]; // the same entries as HBM slots (nullptr unless fyx_enable_instances)
    uint32_t *counts;              // counts[f * kCountStride]
    float one, negzero;            // 1.0f, -0.0f: run-time operands of the unfusable packed FMAs (fyx_math.cuh)
    uint32_t shadow_bits;          // bit f: frustum f is a shadow pass (FYX_PASS_SHADOW)
    uint32_t cam_same;             // non-zero: every frustum of the call has the same camera render mask (f[0].cam_mask)
};

struct SkinArrays {
    // bone table (one entry per (surface, bone))
    uint32_t n_entries;
    const uint32_t *bone_slot; // slot of the bone node, FYX_NONE ⇒ identity
    const float4 *ib[3];       // inverse bind pose rows
    float *palette;            // n_entries * 16 f32, column-major mat4 (the reference's bone_matrices layout)
    // input vertices: blocks of 128 vertices (32 four-vertex groups), 11 rows of 32 float4 (512 B) each:
    //   rows 0-2 position x,y,z   rows 3-5 normal x,y,z   rows 6-9 weight 0..3   row 10 the 4x u8 bone indices;
    // element l of a row belongs to group l of the block and holds the value of its 4 vertices.  A warp reads
    // a row with one perfectly coalesced 512 B access and every 32 B sector exactly once (44 B/vertex).
    const float4 *vblk;
    float *opos, *onrm;        // skinned streams, packed xyz (each surface padded to a multiple of 4 vertices)
    // N4 blend shapes (optional): f16 position / normal offsets per (shape, vertex) in blocks of 128 vertices x 6 rows
    // (px,py,pz,nx,ny,nz) x 32 groups x 4 halfs = 1536 B per (shape, block); weights = BlendShape::weight / 100
    const uint2 *bs;
    const float *bs_w;
    // skinned tangents (optional, per surface; fyx_set_skinned_tangents): tangent xyz in blocks of 128 vertices x 3 rows
    // (tx,ty,tz) of 32 float4 (1536 B), the same row / group convention as vblk but counted from the surface's first
    // vertex; the output otan is one packed-xyz stream per tangent surface (padded to a multiple of 4 vertices).  Their
    // blend-shape offsets (halfs 6-8 of each record) in blocks of 3 rows x 32 groups x 4 halfs = 768 B per (shape, block).
    const float4 *tblk;
    float *otan;
    const uint2 *bst;
};

struct SkinTile {
    uint32_t bone_off; // first palette entry of the surface
    uint32_t n_bones;
    uint32_t quad_start; // absolute index of the first 4-vertex group
    uint32_t n_quads;
    // blend shapes of the surface (n_shapes = 0: none)
    uint32_t n_shapes;
    uint32_t bs_off;      // index of (shape 0, block 0) of the surface in units of 192 uint2 (one 1536-byte shape block)
    uint32_t bs_blocks;   // 128-vertex blocks per shape
    uint32_t w_off;       // first weight in bs_w
    uint32_t local_quad0; // the tile's first group relative to the surface's first group
    // tangents of the surface (tan_blk = FYX_NONE: none)
    uint32_t tan_blk;     // first block of the surface in tblk
    uint32_t tan_quad0;   // first group of the surface in otan (12 floats per group)
    uint32_t bst_off;     // index of (shape 0, block 0) of the surface's tangent offsets, in units of kBstBlockU2
};
static_assert(sizeof(SkinTile) == 48, "SkinTile stays 48 B");
constexpr uint32_t kBsBlockU2 = 6 * 32;  // uint2 per (shape, block)
constexpr uint32_t kBstBlockU2 = 3 * 32; // uint2 per (shape, block) of the tangent offsets
constexpr int kTblkStride = 3 * 32;      // float4 per tangent block of 128 vertices
// records (9 halfs per vertex and layer) -> blocked rows: halfs 0-5 into bs (6 rows), halfs 6-8 into bst (3 rows)
void launch_bs_layout(cudaStream_t s, uint32_t n_verts, uint32_t n_shapes, uint32_t layer_stride, const uint16_t *d_records, uint2 *d_dst, uint32_t bs_blocks);
void launch_bs_tan_layout(cudaStream_t s, uint32_t n_verts, uint32_t n_shapes, uint32_t layer_stride, const uint16_t *d_records, uint2 *d_dst,
                          uint32_t bs_blocks);
// VertexBuffer bytes -> the surface's tangent blocks (tblk points at its first block)
void launch_tan_deinterleave(cudaStream_t s, uint32_t n_verts, const unsigned char *d_bytes, uint32_t stride, uint32_t tangent_offset, float4 *tblk);

struct FoldArrays {
    uint32_t n; // skinned mesh nodes
    const uint32_t *node_slot;
    const uint32_t *bone_begin; // n+1 offsets into bone_slot
    const uint32_t *bone_slot;  // bones of all skinned surfaces of the node, in surface order
    // bones the reference's DFS visits AFTER their mesh contribute the position they had before this update
    // (scene/mesh/mod.rs:676-682 reads the stored value): per entry an index into stale_pos, FYX_NONE = use the new one
    const uint32_t *stale_idx;  // nullptr when no such bone exists
    const float4 *stale_pos;
};

// N2 animation sampling (fyx_anim.cu)
struct AnimTrackDev {
    uint32_t anim;       // owning animation
    uint32_t value_kind; // FYX_TV_*
    uint32_t enabled;
    uint32_t n_curves;
    uint32_t first_key[4]; // offsets into the context-wide key array
    uint32_t n_keys[4];
    float first_loc[4], last_loc[4]; // location of each curve's first / last key (keys are immutable once added): the
                                     // common in-range fetch touches only the remembered span, not the curve's ends
};
struct AnimStateDev {
    float time, speed, slice_start, slice_end;
    uint32_t looped, enabled;
    uint32_t group; // 0 = applied directly (AnimationPlayer, auto_apply); g > 0 = source of blend group g
    float weight;   // its PoseWeight::Constant inside that group
};
struct AnimArrays {
    uint32_t n_tracks, n_anims, n_nodes;
    const fyx_curve_key *keys;
    AnimTrackDev *tracks;
    AnimStateDev *state;
    uint4 *hints;                    // TrackBinding::fetch_hints per track
    float4 *values;                  // sampled value per track
    uint32_t *value_ok;              // fetch returned Some
    const uint32_t *track_bind_kind; // binding | value_kind << 8
    // animated nodes (distinct live targets) and, per node, its tracks in (animation, track) order
    const uint32_t *node_slot;
    const uint32_t *node_begin;
    const uint32_t *node_tracks;
};
void launch_animate(cudaStream_t s, const NodeArrays &a, const AnimArrays &an, fyx_trs *trs_by_slot,
                    const fyx_transform_statics *st_by_slot, float dt, uint32_t *d_err);

// N3 draw-prep (fyx_drawprep.cu): one frustum's visible list -> instances grouped by bundle
struct InstParams {
    uint32_t n;                     // visible entries
    const uint32_t *vis_node;       // the visible list (node indices)
    const uint32_t *vis_slot;       // the same entries as slots
    const uint32_t *bundle_of_slot; // nullptr = every node in bundle 0
    const uint32_t *rank_of_slot;   // pre-order DFS rank (fyx_set_dfs_order); nullptr = node index order
    // surfaces of a node (Mesh::surfaces): ms_range[slot] = (first, count) into ms_bundle / ms_skin; count 0 (or ms_range == nullptr)
    // = ONE surface in the node's bundle id, skinned iff the node has a skinned surface (surf_of_slot)
    const uint2 *ms_range;
    const uint32_t *ms_bundle, *ms_skin;
    const uint32_t *surf_of_slot;   // the node's first skinned fyx surface, FYX_NONE = none
    float view[16], vp[16];         // column-major
    uint32_t n_bundle_ids;
    // scratch (hist and first_key are cleared by the caller: 0 / ~0)
    uint32_t *hist;                 // n_bundle_ids: instances per bundle, then the scatter cursor
    unsigned long long *first_key;  // n_bundle_ids: min (rank << 32 | list position) of the bundle
    uint32_t *offset;               // n_bundle_ids: first instance of the bundle
    uint64_t *tmp_sort;             // n
    // outputs
    uint32_t *o_node;
    uint64_t *o_sort;
    uint32_t *o_surf;               // ordinal of the instance's surface within its node
    uint32_t *o_skin;               // fyx surface id whose palette skins the instance, FYX_NONE = unskinned
    float4 *o_mats;                 // 8 float4 per instance: world (4 columns), view_projection * world (4 columns)
    fyx_bundle *o_bundles;
    uint32_t *o_n_bundles;
};
void launch_inst_count(cudaStream_t s, const NodeArrays &a, const InstParams &ip);   // keys + scan: o_n_bundles[0] = bundles, [2] = instances
void launch_inst_scatter(cudaStream_t s, const NodeArrays &a, const InstParams &ip);
void launch_bone_block_index(cudaStream_t s, uint32_t n, const uint32_t *inst_skin, uint32_t *block_of_inst, uint32_t *counter);
void launch_bone_blocks(cudaStream_t s, uint32_t n, const uint32_t *inst_skin, const uint2 *surf_bones, const float *palette, const uint32_t *block_of_inst,
                        float *blocks);

// Sub-forest plan (fyx_set_topology): the deep levels of the hierarchy — small sub-trees such as skeletons — are cut into groups
// of whole sub-trees; one CTA walks all levels of its group with CTA-wide barriers instead of one kernel launch per level.
// Slots are sorted by (depth, parent slot), so the nodes of a group form ONE contiguous slot range in every level.
constexpr uint32_t kSfCap = 384; // nodes per level and CTA (the previous level's matrices stay in shared memory)
struct SubforestPlan {
    uint32_t n_ctas = 0, n_levels = 0, first_level = 0; // deep levels = [first_level, first_level + n_levels)
    const uint2 *rng = nullptr;                        // [cta][level] = slot range (begin, end)
};
// deferred compaction: the level kernels only store each node's visible bits; this pass turns the bit column into the lists
void launch_compact_vis(cudaStream_t s, const NodeArrays &a, const CullParams &cp);
bool cull_defers_compaction(int nf);
void launch_update_subforest(cudaStream_t s, const NodeArrays &a, const SubforestPlan &sf, bool update_all, const CullParams *cull);

// ---- launchers (fyx_kernels.cu) ----
void launch_update_level(cudaStream_t s, const NodeArrays &a, uint32_t lo, uint32_t hi, bool update_all,
                         const CullParams *cull /* nullptr = no fused cull */);
void launch_cull(cudaStream_t s, const NodeArrays &a, const CullParams &cp, const uint32_t *lodp = nullptr /* per slot: frusta hidden by the LOD filter */);
// one hierarchy level [lo, hi) with DFS pruning by rendered static batches (prune: per slot, frusta hidden for the children)
void launch_cull_range(cudaStream_t s, const NodeArrays &a, const CullParams &cp, const uint32_t *lodp, uint32_t lo, uint32_t hi, uint32_t *prune);
// N4 LOD filter (fyx_drawprep.cu): per observer translation, z_near and z_far - z_near
struct LodParams {
    int nf;
    float ox[FYX_MAX_FRUSTA], oy[FYX_MAX_FRUSTA], oz[FYX_MAX_FRUSTA], zn[FYX_MAX_FRUSTA], zr[FYX_MAX_FRUSTA];
};
void launch_lod_level(cudaStream_t s, const NodeArrays &a, uint32_t lo, uint32_t hi, const float2 *range, uint32_t *lodp, const LodParams &lp);
void launch_select_probes(cudaStream_t s, const NodeArrays &a, const LodParams &obs, uint32_t *best /* [nf], cleared to 0 by the caller: node index + 1 */);
void launch_cull_lights(cudaStream_t s, const NodeArrays &a, const CullParams &cp, uint32_t *const *d_out_ptrs, uint32_t *counts);
void launch_fold_bones(cudaStream_t s, const NodeArrays &a, const FoldArrays &fa, const CullParams *cull);
void launch_snapshot_bones(cudaStream_t s, const NodeArrays &a, uint32_t n_late, const uint32_t *late_slot, float4 *stale_pos);
void launch_palette(cudaStream_t s, const NodeArrays &a, const SkinArrays &sk);
void launch_skin(cudaStream_t s, const SkinArrays &sk, const SkinTile *tiles, uint32_t n_tiles, uint32_t max_bones, bool blend_shapes,
                 bool tangents);

void launch_scatter_locals(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                           const float *d_m16, const uint32_t *slot_of_node, uint32_t n_nodes, uint32_t *d_err);
void launch_scatter_trs(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx, const void *d_payload /* fyx_trs or float4 quats */,
                        bool rot_only, fyx_trs *trs_by_slot /* device copy of the last records; may be nullptr unless rot_only */,
                        const fyx_transform_statics *statics_by_slot /* nullptr = defaults */, const uint32_t *slot_of_node,
                        uint32_t n_nodes, uint32_t *d_err);
void launch_fill_identity_trs(cudaStream_t s, fyx_trs *trs_by_slot, uint32_t n);
void launch_scatter_statics(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                            const fyx_transform_statics *d_in, fyx_transform_statics *statics_by_slot,
                            const uint32_t *slot_of_node, uint32_t n_nodes);
void launch_fill_default_statics(cudaStream_t s, fyx_transform_statics *statics_by_slot, uint32_t n);
void launch_scatter_u32(cudaStream_t s, uint32_t *dst_col, uint32_t count, const uint32_t *d_idx,
                        const uint32_t *d_val, const uint32_t *slot_of_node, uint32_t n_nodes, int mode);
void launch_scatter_aabbs(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                          const float *d_aabb6, const uint32_t *slot_of_node, uint32_t n_nodes);
void launch_gather_globals(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                           const uint32_t *slot_of_node, uint32_t n_nodes, float *d_out_m16);
void launch_gather_aabbs(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                         const uint32_t *slot_of_node, uint32_t n_nodes, float *d_out6);
void launch_gather_flags(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                         const uint32_t *slot_of_node, uint32_t n_nodes, uint32_t *d_out);
void launch_deinterleave(cudaStream_t s, uint32_t n_verts, const unsigned char *d_bytes, fyx_vertex_layout layout,
                         uint32_t n_bones, float4 *vblk, uint64_t first_vertex, uint32_t *d_err);
constexpr int kVblkRows = 11;                    // float4 rows per block
constexpr int kVblkStride = kVblkRows * 32;      // float4 per block of 128 vertices
void launch_ib_rows(cudaStream_t s, uint32_t n, const float *d_m16, float4 *r0, float4 *r1, float4 *r2, uint32_t *d_err);
void launch_or_u32(cudaStream_t s, uint32_t *p, uint32_t bits);
// dst[s] = map[s] != FYX_NONE ? src[map[s]] : default, records of `words` 32-bit words (<= 32): carries per-slot data over a
// topology change (slots move; fyx_set_topology)
struct PermuteDefault { uint32_t w[32]; };
void launch_permute_words(cudaStream_t s, void *dst, const void *src, const uint32_t *map, uint32_t n, uint32_t words, const PermuteDefault &def);
void launch_compact_gathered(cudaStream_t s, const uint32_t *pad, uint32_t maxc, const uint32_t *counts_all, int nranks, int f,
                             uint32_t *dst);

// ---- multi-GPU exchange by peer stores (fyx_peer.cu) ----
constexpr int kPeerMaxRanks = 16;
struct PeerCtrl { // lives at the start of every rank's exchange allocation; written by the peers
    uint32_t counts[2][kPeerMaxRanks][FYX_MAX_FRUSTA]; // [epoch & 1][rank][frustum]
    uint32_t cnt_flag[2][kPeerMaxRanks];               // epoch of rank r's last count publication
    uint32_t done_flag[2][kPeerMaxRanks];              // epoch of rank r's last completed push into THIS rank's lists
    uint32_t totals[2][FYX_MAX_FRUSTA];                // gathered count per frustum (written by k_peer_wait)
};
constexpr size_t kPeerCtrlBytes = 4096;
static_assert(sizeof(PeerCtrl) <= kPeerCtrlBytes, "control block fits its page");
struct PeerParams {
    int nranks, rank, nf;
    uint32_t epoch;
    unsigned char *base[kPeerMaxRanks]; // every rank's exchange allocation as mapped into this process
    uint64_t total_cap;                 // entries per (slot, frustum) list: all ranks' slots together
    uint32_t nf_cap;
    const uint32_t *own_list[FYX_MAX_FRUSTA];
    const uint32_t *own_counts; // counts[f * kCountStride]
    uint32_t *cta_done;
    uint32_t *d_err;
};
__host__ __device__ inline PeerCtrl *peer_ctrl(const PeerParams &pp, int r) { return reinterpret_cast<PeerCtrl *>(pp.base[r]); }
__host__ __device__ inline uint32_t *peer_list(const PeerParams &pp, int r, uint32_t slot, uint32_t f)
{
    return reinterpret_cast<uint32_t *>(pp.base[r] + kPeerCtrlBytes) + ((size_t)slot * pp.nf_cap + f) * pp.total_cap;
}
void launch_peer_counts(cudaStream_t s, const PeerParams &pp);                   // publish this rank's counts, wait for everybody's
void launch_peer_push(cudaStream_t s, const PeerParams &pp, unsigned push_ctas); // store the lists into every rank's buffers, wait for everybody's

// error bits written by kernels into d_err
constexpr uint32_t E_NOT_AFFINE = 1u;
constexpr uint32_t E_BAD_BONE_INDEX = 2u;
constexpr uint32_t E_NONFINITE_VERTEX = 4u;
constexpr uint32_t E_PEER_TIMEOUT = 8u; // a rank never showed up in the peer exchange (bounded spin, fyx_peer.cu)

} // namespace fyx
