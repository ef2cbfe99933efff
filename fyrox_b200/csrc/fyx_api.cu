// fyx_api.cu — the C ABI of libfyrox_b200 (include/fyrox_b200.h): context, host-side bookkeeping
// (slot ordering by hierarchy depth, staging, surface tables) and stream-ordered kernel launches.
// No CPU fallback exists: every compute entry point launches the sm_100a kernels of fyx_kernels.cu.
#include <algorithm>
#include <limits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "fyx_hostseg.hpp"
#include "fyx_internal.h"

using namespace fyx;

// --------------------------------------------------------------------------------------------
// small utilities
// --------------------------------------------------------------------------------------------
namespace {

thread_local std::string g_create_error;

struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    template <class T> T *as() const { return static_cast<T *>(p); }
};

struct Surface {
    uint32_t mesh_node;
    uint32_t n_bones;
    uint32_t bone_off;  // first palette entry
    uint32_t n_verts;
    uint64_t vert_off;  // first vertex (multiple of 4)
    std::vector<uint32_t> bones; // node indices
    // N4 blend shapes
    uint32_t n_shapes = 0, bs_blocks = 0, bs_cap = 0; // shapes, 128-vertex blocks per shape, capacity of the region in shape blocks
    uint64_t bs_off = 0;                               // first shape block of the region
    uint32_t w_off = 0, w_cap = 0;
    // skinned tangents (fyx_set_skinned_tangents): on, and the surface's regions (kept when turned off, reused when turned on again)
    bool tangents = false;
    uint32_t tan_blk = FYX_NONE;  // first block in b_tblk
    uint32_t tan_quad0 = 0;       // first 4-vertex group in b_otan
    uint32_t bst_off = 0, bst_cap = 0; // tangent blend-shape region in b_bst: first shape block, capacity in shape blocks
};

enum { EV_START = 0, EV_UPLOAD, EV_UPDATE, EV_CULL, EV_PALETTE, EV_SKIN, EV_READBACK, EV_COUNT };

// Output of one cull: per-frustum visible lists + counters, device and (pinned) host side.  Two slots
// alternate so that the lists of frame i can travel to the host while frame i+1 is being culled.
struct VisSlot {
    DevBuf b_vis[FYX_MAX_FRUSTA];
    DevBuf b_vis_slot[FYX_MAX_FRUSTA]; // the same entries as HBM slots (fyx_enable_instances)
    bool have_slots = false;
    uint32_t *d_counts = nullptr; // kCountStride * FYX_MAX_FRUSTA, each counter on its own 128 B line
    uint32_t *h_counts = nullptr; // pinned, FYX_MAX_FRUSTA
    uint32_t *h_vis[FYX_MAX_FRUSTA] = {};
    size_t h_vis_cap[FYX_MAX_FRUSTA] = {};
    uint32_t nf = 0;
    bool counts_on_host = false, lists_on_host = false;
    // multi-GPU: the all-gathered lists of this frame (padded slots, packed list, host copy)
    DevBuf b_gath_pad[FYX_MAX_FRUSTA], b_gath[FYX_MAX_FRUSTA];
    uint32_t gath_count[FYX_MAX_FRUSTA] = {};
    uint32_t *h_gath[FYX_MAX_FRUSTA] = {};
    size_t h_gath_cap[FYX_MAX_FRUSTA] = {};
    bool gathered = false, gathered_on_host = false;
    bool own_only = false; // FYX_FRAME_READBACK_OWN: the host copy of this frame is the rank's own lists
    cudaEvent_t ev_gather = nullptr, ev_counts_all = nullptr;
    uint64_t epoch = 0;            // number of this gathered frame (the same on every rank)
    bool via_peer = false;         // exchanged by peer stores (fyx_peer.cu), else NCCL
    uint32_t *gath_ptr[FYX_MAX_FRUSTA] = {}; // the gathered list on the device (peer allocation or b_gath)
    uint32_t counts_all[kPeerMaxRanks][FYX_MAX_FRUSTA] = {};
    bool counts_all_known = false;
    // host copy of the gathered lists through the node-wide segment (fyx_hostseg.hpp)
    bool host_copy_private = false; // the frame did not ask for a read-back: a later fetch copies the device list privately
    bool seg_published = false, seg_complete = false, own_in_seg = false;
    uint32_t *seg_own[FYX_MAX_FRUSTA] = {};
    bool pending = false; // written by a pipelined (async + read-back) frame that fyx_frame_wait has not collected yet
    uint64_t frame_no = 0;
    cudaEvent_t ev_cull = nullptr, ev_counts = nullptr, ev_done = nullptr;
};

// N2: one animation on the host side (fyx_anim.inl)
struct AnimHost {
    uint32_t first_track = 0, n_tracks = 0, pos_in_group = 0;
    AnimStateDev st{};
};

// N3: packed instances of one frustum (fyx_drawprep.inl)
struct InstOut {
    DevBuf b_node, b_sort, b_mats, b_bundles, b_surf, b_skin;
    void *h_surf = nullptr;
    size_t h_surf_cap = 0;
    uint32_t n_visible = 0;
    DevBuf b_block_of, b_blocks; // bone-matrix blocks of the skinned instances (fyx_pack_bone_matrices)
    uint32_t n_blocks = 0;
    bool blocks_valid = false;
    void *h[4] = {};
    size_t h_cap[4] = {};
    uint32_t count = 0, n_bundles = 0;
    bool valid = false, on_host = false;
};

} // namespace

struct PeerState {
    void *local = nullptr;                 // this rank's exchange allocation (control block + 2 x F lists)
    void *mapped[kPeerMaxRanks] = {};      // the other ranks' allocations (cudaIpcOpenMemHandle)
    uint32_t *cta_done = nullptr;
    uint32_t *h_counts = nullptr;          // pinned: [epoch & 1][2][rank][frustum] copy of the count table
    PeerParams pp{};
    bool ready = false;
};

struct fyx_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    uint64_t launches = 0;

    // topology
    uint32_t n_nodes = 0, n_slots = 0, root = FYX_NONE, n_renderable = 0;
    std::vector<uint32_t> slot_of_node, node_of_slot, level_off;
    NodeArrays a{};
    DevBuf b_vis;
    DevBuf b_parent, b_flags, b_mask, b_gidx, b_L[3], b_G[3], b_la[3], b_wa[3], b_slot_of_node;
    bool have_topology = false, updated_once = false;
    SubforestPlan sf{};  // deep levels walked by one launch (fyx_internal.h); n_ctas = 0: one launch per level everywhere
    DevBuf b_sf_rng;
    DevBuf b_statics; // fyx_transform_statics per slot, allocated by the first fyx_set_transform_statics
    bool have_statics = false;
    DevBuf b_trs;     // fyx_trs per slot: the last position/rotation/scale sent for each node (first TRS call allocates)
    bool have_trs = false;

    // error word written by kernels
    uint32_t *d_err = nullptr;
    uint32_t *h_err = nullptr; // pinned

    // staging (host pinned + device)
    void *h_stage = nullptr;
    size_t h_stage_bytes = 0;
    DevBuf d_stage;

    // cull outputs
    CullParams cp{};
    VisSlot vs[2];
    int cur = 0;      // slot written by the most recent cull
    int readable = 0; // slot fyx_get_visible reads
    uint64_t frame_counter = 0;

    // frame pipelining (FYX_FRAME_ASYNC): uploads on their own stream into alternating staging buffers,
    // read-backs on a third stream
    cudaStream_t copy_stream = nullptr, d2h_stream = nullptr;
    cudaStream_t fold_stream = nullptr; // skinned-mesh fold + cull beside the palette / skinning kernels of asynchronous frames
    cudaEvent_t ev_levels_done = nullptr, ev_fold_done = nullptr;
    DevBuf d_stage_frame[2];
    cudaEvent_t ev_upload[2] = {}, ev_slot_free[2] = {};
    bool slot_used[2] = {false, false};
    int upload_parity = 0;
    cudaEvent_t ev_levels_prev = nullptr; // the previous frame's "level kernels + fold + cull are done" event (its ev_cull), if it recorded one
    uint64_t launches_at_frame_end = ~0ull;

    // skinning
    std::vector<Surface> surfaces;
    bool tables_dirty = false;
    uint64_t n_verts_total = 0; // padded
    uint64_t vert_cap = 0;
    uint32_t n_entries = 0, entry_cap = 0;
    DevBuf b_vblk, b_opos, b_onrm, b_ib[3], b_palette, b_bone_slot, b_tiles;
    // surfaces per node (fyx_set_node_surfaces): host CSR by node, device table by slot (rebuilt when dirty)
    std::vector<uint2> ms_of_node;       // (first, count) into ms_bundle_h / ms_skin_h; count 0 = default single surface
    std::vector<uint32_t> ms_bundle_h, ms_skin_h;
    bool ms_dirty = false, have_ms = false;
    DevBuf b_ms_range, b_ms_bundle, b_ms_skin;
    DevBuf b_surf_of_slot, b_surf_bones; // per slot: the node's first skinned surface (FYX_NONE = none); per surface: (first palette entry, n_bones)
    DevBuf b_bs, b_bs_w;          // blend-shape offsets (blocked f16) and weights
    uint64_t bs_used = 0;         // shape blocks handed out
    uint32_t bs_w_used = 0;
    bool any_blend_shapes = false;
    DevBuf b_tblk, b_otan, b_bst; // skinned tangents: input blocks, output stream, blend-shape offsets (only tangent surfaces have any)
    uint64_t tan_blocks_used = 0, tan_quads_used = 0, bst_used = 0;
    bool any_tangents = false;
    DevBuf b_fold_node, b_fold_begin, b_fold_bone, b_fold_stale_idx, b_late_slot, b_stale_pos;
    std::vector<uint32_t> dfs_rank; // optional: pre-order rank of every node in the reference's DFS (fyx_set_dfs_order)
    uint32_t n_late = 0;
    uint32_t n_tiles = 0, max_bones = 0;
    FoldArrays fold{};
    SkinArrays sk{};
    std::vector<uint8_t> skinned_node; // per node: has a skinned surface

    // timing
    cudaEvent_t ev[EV_COUNT] = {};
    fyx_timings timings{};
    bool timings_pending = false; // an async frame's events have not been read yet
    bool stage_events_valid = false; // the last frame recorded the per-stage events (synchronous frames only)

    // N2 animation sampling (fyx_anim.inl)
    std::vector<AnimHost> anims;
    std::vector<fyx_anim_track> anim_tracks; // all tracks, animation after animation
    uint32_t n_anim_keys = 0, n_blend_groups = 0;
    std::vector<std::vector<uint32_t>> blend_groups; // sources of group g at [g - 1]
    bool anim_csr_dirty = true;
    std::vector<fyx_curve_key> pend_keys; // queued by fyx_anim_add, uploaded by anim_flush
    std::vector<AnimTrackDev> pend_tracks;
    std::vector<uint32_t> pend_bk;
    std::vector<AnimStateDev> pend_state;
    AnimArrays an{};
    DevBuf b_anim_keys, b_anim_tracks, b_anim_state, b_anim_hints, b_anim_values, b_anim_ok, b_anim_bk, b_anim_node_slot,
        b_anim_node_begin, b_anim_node_tracks;

    // N4 LOD filter (fyx_drawprep.inl)
    DevBuf b_lod_range, b_lodp; // float2 (begin, end; begin NaN = not a LOD object) and hidden-frusta bits, per slot
    DevBuf b_prune;             // per slot: frusta in which the node's children are pruned (rendered static batches, hidden ancestors)
    bool maybe_static_batch = false; // some node carries FYX_NODE_STATIC_BATCH: the cull runs level by level
    bool have_lod = false;
    std::vector<fyx_observer> observers;

    // N4 light lists (fyx_drawprep.inl)
    DevBuf b_light[FYX_MAX_FRUSTA], b_light_ptrs, b_light_counts;
    uint32_t *h_light_counts = nullptr; // pinned
    std::vector<uint32_t> h_light[FYX_MAX_FRUSTA];
    uint32_t light_nf = 0;
    bool lights_valid = false;

    // N3 draw-prep (fyx_drawprep.inl)
    bool instances_enabled = false, have_bundles = false, rank_on_device = false;
    uint32_t n_bundle_ids = 1;
    DevBuf b_bundle, b_rank_slot, b_inst_hist, b_inst_first, b_inst_offset, b_inst_tmp, b_inst_nb;
    uint32_t *h_inst_nb = nullptr;
    InstOut inst[FYX_MAX_FRUSTA];

    // multi-GPU (fyx_comm.cu)
    void *comm = nullptr;
    int nranks = 1, rank = 0;
    cudaStream_t comm_stream = nullptr; // the collective runs beside the palette / skinning kernels (highest priority)
    DevBuf b_counts_packed, b_counts_all;
    uint32_t *h_counts_all = nullptr; // pinned nranks*FYX_MAX_FRUSTA
    bool want_peer = true, want_hostseg = true;
    unsigned peer_push_ctas = 96;
    bool exchange_built = false, hostseg_ready = false, hostseg_registered = false;
    uint32_t exchange_slots = 0, exch_nf_cap = 0;
    uint64_t exch_total_cap = 0, gather_epoch = 0;
    PeerState peer;
    HostSeg hostseg;
    cudaEvent_t ev_x0[2] = {}, ev_x1[2] = {}; // timing of the exchange (per epoch parity)
    uint64_t x_epoch[2] = {0, 0};
    int x_slot[2] = {0, 0};
    cudaEvent_t ev_gath_read[2] = {}; // private D2H copies of the gathered device lists (per epoch parity)
    bool gath_read_valid[2] = {false, false};
};

namespace {

int32_t fail(fyx_ctx *c, int32_t code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    else g_create_error = buf;
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            return fail(c, e__ == cudaErrorMemoryAllocation ? FYX_ERR_OUT_OF_MEMORY : FYX_ERR_CUDA,      \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__);    \
    } while (0)

int32_t dev_ensure(fyx_ctx *c, DevBuf &b, size_t bytes, bool keep = false)
{
    if (bytes <= b.bytes) return FYX_OK;
    size_t nb = keep ? std::max(bytes, b.bytes + b.bytes / 2) : bytes;
    nb = (nb + 255) & ~size_t(255);
    void *np = nullptr;
    CU(cudaMalloc(&np, nb));
    // growable tables are copied as a whole when they grow again: give their not-yet-written tail a defined value
    if (keep) CU(cudaMemsetAsync(np, 0, nb, c->stream));
    if (b.p) {
        cudaError_t e = cudaSuccess;
        if (keep && b.bytes) e = cudaMemcpyAsync(np, b.p, b.bytes, cudaMemcpyDeviceToDevice, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) {
            cudaFree(np); // the old buffer stays valid
            return fail(c, FYX_ERR_CUDA, "growing a device buffer failed: %s", cudaGetErrorString(e));
        }
        cudaFree(b.p);
    }
    b.p = np;
    b.bytes = nb;
    return FYX_OK;
}

void dev_free(DevBuf &b)
{
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
}

int32_t host_stage_ensure(fyx_ctx *c, size_t bytes)
{
    if (bytes <= c->h_stage_bytes) return FYX_OK;
    if (c->h_stage) {
        CU(cudaStreamSynchronize(c->stream));
        cudaFreeHost(c->h_stage);
        c->h_stage = nullptr;
        c->h_stage_bytes = 0;
    }
    size_t nb = (bytes + bytes / 4 + 4095) & ~size_t(4095);
    CU(cudaHostAlloc(&c->h_stage, nb, cudaHostAllocDefault));
    c->h_stage_bytes = nb;
    return FYX_OK;
}

bool is_pinned(const void *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

// Host → device staging of one or two arrays.  `direct` lets pinned caller memory be DMA'd without
// the bounce copy (only legal when the caller's buffer stays untouched until the next sync, i.e.
// inside fyx_render_prep).  Returns device pointers inside d_stage.
int32_t stage_to_device(fyx_ctx *c, const void *a0, size_t n0, const void *a1, size_t n1, bool direct, void **d0, void **d1)
{
    const size_t o1 = (n0 + 255) & ~size_t(255);
    const size_t total = o1 + ((n1 + 255) & ~size_t(255));
    int32_t rc = dev_ensure(c, c->d_stage, total);
    if (rc) return rc;
    char *dbase = c->d_stage.as<char>();
    const void *src[2] = {a0, a1};
    const size_t len[2] = {n0, n1};
    const size_t off[2] = {0, o1};
    bool need_bounce = false;
    for (int i = 0; i < 2; ++i)
        if (src[i] && len[i] && !(direct && is_pinned(src[i]))) need_bounce = true;
    if (need_bounce) {
        rc = host_stage_ensure(c, total);
        if (rc) return rc;
        // the previous use of the bounce buffer must have drained
        CU(cudaStreamSynchronize(c->stream));
    }
    for (int i = 0; i < 2; ++i) {
        if (!src[i] || !len[i]) continue;
        const void *from = src[i];
        if (!(direct && is_pinned(src[i]))) {
            memcpy(static_cast<char *>(c->h_stage) + off[i], src[i], len[i]);
            from = static_cast<char *>(c->h_stage) + off[i];
        }
        CU(cudaMemcpyAsync(dbase + off[i], from, len[i], cudaMemcpyHostToDevice, c->stream));
    }
    *d0 = (a0 && n0) ? dbase : nullptr;
    if (d1) *d1 = (a1 && n1) ? dbase + o1 : nullptr;
    return FYX_OK;
}

int32_t check_device_errors(fyx_ctx *c)
{
    // called right after a stream synchronisation; h_err was copied before it
    const uint32_t e = *c->h_err;
    if (!e) return FYX_OK;
    *c->h_err = 0;
    cudaMemsetAsync(c->d_err, 0, sizeof(uint32_t), c->stream);
    if (e & E_NOT_AFFINE)
        return fail(c, FYX_ERR_NOT_AFFINE, "a matrix with a bottom row other than (0,0,0,1) or a non-finite entry was skipped");
    if (e & E_BAD_BONE_INDEX) return fail(c, FYX_ERR_INVALID_ARGUMENT, "a vertex references a bone index >= n_bones");
    if (e & E_NONFINITE_VERTEX) return fail(c, FYX_ERR_INVALID_ARGUMENT, "a vertex position is not finite");
    if (e & E_PEER_TIMEOUT) return fail(c, FYX_ERR_NCCL, "the peer exchange of the visible lists timed out: a rank did not take part in the frame");
    return FYX_OK;
}

int32_t sync_and_check(fyx_ctx *c)
{
    CU(cudaMemcpyAsync(c->h_err, c->d_err, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaGetLastError());
    return check_device_errors(c);
}

void rebuild_node_arrays(fyx_ctx *c)
{
    NodeArrays &a = c->a;
    a.cap = c->n_slots;
    a.parent = c->b_parent.as<uint32_t>();
    a.flags = c->b_flags.as<uint32_t>();
    a.mask = c->b_mask.as<uint32_t>();
    a.gidx = c->b_gidx.as<uint32_t>();
    a.vis = c->b_vis.as<uint8_t>();
    for (int i = 0; i < 3; ++i) {
        a.L[i] = c->b_L[i].as<float4>();
        a.G[i] = c->b_G[i].as<float4>();
        a.la[i] = c->b_la[i].as<float2>();
        a.wa[i] = c->b_wa[i].as<float2>();
    }
}

// Frustum → kernel parameter form
void to_dev_frustum(const fyx_frustum &f, uint32_t cam_mask, uint32_t pass_flags, FrustumDev &d)
{
    for (int p = 0; p < 6; ++p) d.plane[p] = make_float4(f.planes[p][0], f.planes[p][1], f.planes[p][2], f.planes[p][3]);
    for (int i = 0; i < 8; ++i) d.corner[i] = make_float4(f.corners[i][0], f.corners[i][1], f.corners[i][2], 0.0f);
    for (int q = 0; q < 3; ++q)
        for (int k = 0; k < 4; ++k) d.pn[q][k] = make_float2(f.planes[2 * q][k], f.planes[2 * q + 1][k]);
    // distinct corner coordinates per axis (bit-pattern equality, so -0/+0 and NaNs stay separate entries:
    // each entry is compared exactly like the corner it came from)
    d.n_ax = 0;
    for (int k = 0; k < 3; ++k) {
        int n = 0;
        uint32_t masks[8] = {0};
        float vals[8];
        for (int j = 0; j < 8; ++j) d.ax_mask[k][j] = 0;
        for (int i = 0; i < 8; ++i) {
            const float v = f.corners[i][k];
            uint32_t vb, ub;
            memcpy(&vb, &v, 4);
            int j = 0;
            for (; j < n; ++j) {
                memcpy(&ub, &vals[j], 4);
                if (ub == vb) break;
            }
            if (j == n) {
                vals[n] = v;
                ++n;
            }
            masks[j] |= 1u << i;
        }
        for (int j = n; j < 8; ++j) vals[j] = std::nanf(""); // never inside any box
        d.ax_val[k][0] = make_float4(vals[0], vals[1], vals[2], vals[3]);
        d.ax_val[k][1] = make_float4(vals[4], vals[5], vals[6], vals[7]);
        for (int j = 0; j < n; ++j) d.ax_mask[k][j] = masks[j];
        d.n_ax |= (uint32_t)n << (8 * k);
    }
    d.cam_mask = cam_mask;
    d.pass_flags = pass_flags;
    for (int p = 0; p < 6; ++p)
        for (int k = 0; k < 3; ++k) d.vsel[p >> 1][k][p & 1] = (f.planes[p][k] < 0.0f) ? 0x3210u : 0x7654u;
    // smallest plane value over the frustum's own corners, one rounding per operation in the kernels' order (the volatile
    // temporaries keep the host compiler from contracting anything)
    for (int p = 0; p < 6; ++p) {
        float m = std::numeric_limits<float>::infinity();
        for (int i = 0; i < 8; ++i) {
            volatile float a = f.planes[p][0] * f.corners[i][0];
            volatile float b = f.planes[p][1] * f.corners[i][1];
            volatile float ab = a + b;
            volatile float e = f.planes[p][2] * f.corners[i][2];
            volatile float abe = ab + e;
            volatile float sv = abe + f.planes[p][3];
            const float v = sv;
            if (std::isnan(v) || std::isnan(m)) m = std::nanf("");
            else if (v < m) m = v;
        }
        if (p & 1) d.pm[p >> 1].y = m;
        else d.pm[p >> 1].x = m;
    }
}

int32_t prepare_cull(fyx_ctx *c, uint32_t nf, const fyx_frustum *fr, const uint32_t *cam_mask, const uint32_t *pass_flags)
{
    if (nf > FYX_MAX_FRUSTA) return fail(c, FYX_ERR_INVALID_ARGUMENT, "n_frusta %u > FYX_MAX_FRUSTA", nf);
    if (nf && !fr) return fail(c, FYX_ERR_INVALID_ARGUMENT, "frusta is NULL");
    const int slot = c->cur ^ 1;
    VisSlot &V = c->vs[slot];
    if (V.pending) return fail(c, FYX_ERR_STATE, "two pipelined frames are already in flight: call fyx_frame_wait first");
    c->cur = slot;
    c->cp.nf = (int)nf;
    c->cp.counts = V.d_counts;
    c->cp.one = 1.0f;
    c->cp.negzero = -0.0f;
    c->cp.shadow_bits = 0u;
    c->cp.cam_same = 1u;
    for (uint32_t f = 0; f < nf; ++f) {
        to_dev_frustum(fr[f], cam_mask ? cam_mask[f] : 0xFFFFFFFFu, pass_flags ? pass_flags[f] : 0u, c->cp.f[f]);
        if (c->cp.f[f].pass_flags & FYX_PASS_SHADOW) c->cp.shadow_bits |= 1u << f;
        if (c->cp.f[f].cam_mask != c->cp.f[0].cam_mask) c->cp.cam_same = 0u;
        // worst case every alive node is visible (fyx_set_flags may turn any of them renderable)
        int32_t rc = dev_ensure(c, V.b_vis[f], sizeof(uint32_t) * std::max<size_t>(c->n_slots, 1));
        if (rc) return rc;
        c->cp.out[f] = V.b_vis[f].as<uint32_t>();
        c->cp.out_slot[f] = nullptr;
        if (c->instances_enabled) {
            rc = dev_ensure(c, V.b_vis_slot[f], sizeof(uint32_t) * std::max<size_t>(c->n_slots, 1));
            if (rc) return rc;
            c->cp.out_slot[f] = V.b_vis_slot[f].as<uint32_t>();
        }
    }
    V.have_slots = c->instances_enabled;
    for (auto &o : c->inst) o.valid = false;
    c->lights_valid = false;
    CU(cudaMemsetAsync(V.d_counts, 0, sizeof(uint32_t) * kCountStride * FYX_MAX_FRUSTA, c->stream));
    V.nf = nf;
    V.counts_on_host = V.lists_on_host = false;
    V.gathered = V.gathered_on_host = false;
    V.seg_published = V.seg_complete = V.own_in_seg = V.counts_all_known = V.host_copy_private = false;
    c->readable = slot;
    return FYX_OK;
}

// Hierarchy + boxes (+ fused cull): one launch per level (parents first), then the skinned-mesh fold.
// fold_on: stream for the skinned-mesh fold (+ cull of the skinned meshes); nullptr = the main stream, in order.  Another stream
// is given by asynchronous frames that go on to the palette / skinning kernels: those need the bones' matrices, not the meshes'
// boxes, so the (latency-bound) fold runs beside them; the caller joins the streams.
int32_t run_update(fyx_ctx *c, uint32_t update_flags, const CullParams *cull, cudaStream_t fold_on = nullptr)
{
    const bool all = (update_flags & FYX_UPDATE_ALL) || !c->updated_once;
    const size_t nl = c->level_off.size() ? c->level_off.size() - 1 : 0;
    if (c->n_late) {
        launch_snapshot_bones(c->stream, c->a, c->n_late, c->b_late_slot.as<uint32_t>(), c->b_stale_pos.as<float4>());
        c->launches++;
    }
    const size_t nl_wide = c->sf.n_ctas ? std::min<size_t>(nl, c->sf.first_level) : nl;
    for (size_t l = 0; l < nl_wide; ++l) {
        launch_update_level(c->stream, c->a, c->level_off[l], c->level_off[l + 1], all, cull);
        c->launches += (c->level_off[l + 1] > c->level_off[l]);
    }
    if (c->sf.n_ctas) { // the deep levels (small sub-trees: skeletons) in one launch
        launch_update_subforest(c->stream, c->a, c->sf, all, cull);
        c->launches++;
    }
    if (cull && cull_defers_compaction(cull->nf)) { // the level kernels stored visible bits: build the lists now
        launch_compact_vis(c->stream, c->a, *cull);
        c->launches++;
    }
    if (c->fold.n) {
        if (fold_on) {
            CU(cudaEventRecord(c->ev_levels_done, c->stream));
            CU(cudaStreamWaitEvent(fold_on, c->ev_levels_done, 0));
        }
        launch_fold_bones(fold_on ? fold_on : c->stream, c->a, c->fold, cull);
        c->launches++;
        if (fold_on) CU(cudaEventRecord(c->ev_fold_done, fold_on));
    }
    c->updated_once = true;
    CU(cudaGetLastError());
    return FYX_OK;
}

int32_t commit_surfaces(fyx_ctx *c);

int32_t host_list_ensure(fyx_ctx *c, VisSlot &V, uint32_t f, size_t n)
{
    if (n <= V.h_vis_cap[f]) return FYX_OK;
    if (V.h_vis[f]) cudaFreeHost(V.h_vis[f]);
    V.h_vis[f] = nullptr;
    const size_t cap = std::max<size_t>(1024, n + n / 2);
    CU(cudaHostAlloc(reinterpret_cast<void **>(&V.h_vis[f]), cap * sizeof(uint32_t), cudaHostAllocDefault));
    V.h_vis_cap[f] = cap;
    return FYX_OK;
}

int32_t host_gath_ensure(fyx_ctx *c, VisSlot &V, uint32_t f, size_t n)
{
    if (n <= V.h_gath_cap[f]) return FYX_OK;
    if (V.h_gath[f]) cudaFreeHost(V.h_gath[f]);
    V.h_gath[f] = nullptr;
    const size_t cap = std::max<size_t>(1024, n + n / 2);
    CU(cudaHostAlloc(reinterpret_cast<void **>(&V.h_gath[f]), cap * sizeof(uint32_t), cudaHostAllocDefault));
    V.h_gath_cap[f] = cap;
    return FYX_OK;
}

// counts, then the lists sized by them, to pinned host memory (stream `s`, two synchronisations)
int32_t readback_visible(fyx_ctx *c, VisSlot &V, cudaStream_t s)
{
    const uint32_t nf = V.nf;
    if (!nf) return FYX_OK;
    if (!V.counts_on_host) {
        CU(cudaMemcpy2DAsync(V.h_counts, sizeof(uint32_t), V.d_counts, sizeof(uint32_t) * kCountStride, sizeof(uint32_t), nf,
                             cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        V.counts_on_host = true;
    }
    if (!V.lists_on_host) {
        for (uint32_t f = 0; f < nf; ++f) {
            const size_t n = V.h_counts[f];
            int32_t rc = host_list_ensure(c, V, f, n);
            if (rc) return rc;
            if (n) CU(cudaMemcpyAsync(V.h_vis[f], V.b_vis[f].p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        }
        CU(cudaStreamSynchronize(s));
        V.lists_on_host = true;
    }
    return FYX_OK;
}

} // namespace

// --------------------------------------------------------------------------------------------
// life cycle
// --------------------------------------------------------------------------------------------
extern "C" uint32_t fyx_abi_version(void) { return FYX_ABI_VERSION; }

extern "C" const char *fyx_last_error(const fyx_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int32_t fyx_create(const fyx_config *cfg, fyx_ctx **out_ctx)
{
    fyx_ctx *c = nullptr; // for CU(): errors before the context exists go to the thread-local string
    if (!out_ctx) return fail(nullptr, FYX_ERR_INVALID_ARGUMENT, "out_ctx is NULL");
    *out_ctx = nullptr;
    int dev = -1;
    void *stream = nullptr;
    if (cfg) {
        if (cfg->struct_size < sizeof(fyx_config)) return fail(nullptr, FYX_ERR_INVALID_ARGUMENT, "fyx_config.struct_size too small");
        dev = cfg->device;
        stream = cfg->stream;
    }
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, FYX_ERR_CUDA, "no CUDA device available (%s): libfyrox_b200 has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (dev < 0) CU(cudaGetDevice(&dev));
    if (dev >= count) return fail(nullptr, FYX_ERR_INVALID_ARGUMENT, "device %d out of range (%d devices)", dev, count);
    CU(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10)
        return fail(nullptr, FYX_ERR_CUDA, "device %d is sm_%d%d; this library ships sm_100a code only", dev, prop.major, prop.minor);

    fyx_ctx *ctx = new (std::nothrow) fyx_ctx();
    if (!ctx) return fail(nullptr, FYX_ERR_OUT_OF_MEMORY, "host allocation failed");
    c = ctx;
    c->device = dev;
    auto bail = [&](int32_t rc) {
        g_create_error = c->err;
        fyx_destroy(c);
        return rc;
    };
#define CUB(call)                                                                                   \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            fail(c, FYX_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__));                 \
            return bail(FYX_ERR_CUDA);                                                              \
        }                                                                                           \
    } while (0)
    if (stream) {
        c->stream = static_cast<cudaStream_t>(stream);
    } else {
        CUB(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
    }
    CUB(cudaMalloc(reinterpret_cast<void **>(&c->d_err), sizeof(uint32_t)));
    CUB(cudaMemset(c->d_err, 0, sizeof(uint32_t)));
    CUB(cudaHostAlloc(reinterpret_cast<void **>(&c->h_err), sizeof(uint32_t), cudaHostAllocDefault));
    *c->h_err = 0;
    for (VisSlot &V : c->vs) {
        CUB(cudaMalloc(reinterpret_cast<void **>(&V.d_counts), sizeof(uint32_t) * kCountStride * FYX_MAX_FRUSTA));
        CUB(cudaMemset(V.d_counts, 0, sizeof(uint32_t) * kCountStride * FYX_MAX_FRUSTA));
        CUB(cudaHostAlloc(reinterpret_cast<void **>(&V.h_counts), sizeof(uint32_t) * FYX_MAX_FRUSTA, cudaHostAllocDefault));
        memset(V.h_counts, 0, sizeof(uint32_t) * FYX_MAX_FRUSTA);
        CUB(cudaEventCreateWithFlags(&V.ev_cull, cudaEventDisableTiming));
        CUB(cudaEventCreateWithFlags(&V.ev_counts, cudaEventDisableTiming));
        CUB(cudaEventCreateWithFlags(&V.ev_done, cudaEventDisableTiming));
        CUB(cudaEventCreateWithFlags(&V.ev_gather, cudaEventDisableTiming));
        CUB(cudaEventCreateWithFlags(&V.ev_counts_all, cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; ++i) {
        CUB(cudaEventCreateWithFlags(&c->ev_gath_read[i], cudaEventDisableTiming));
        CUB(cudaEventCreate(&c->ev_x0[i]));
        CUB(cudaEventCreate(&c->ev_x1[i]));
    }
    CUB(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    CUB(cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
    CUB(cudaStreamCreateWithFlags(&c->fold_stream, cudaStreamNonBlocking));
    CUB(cudaEventCreateWithFlags(&c->ev_levels_done, cudaEventDisableTiming));
    CUB(cudaEventCreateWithFlags(&c->ev_fold_done, cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) {
        CUB(cudaEventCreateWithFlags(&c->ev_upload[i], cudaEventDisableTiming));
        CUB(cudaEventCreateWithFlags(&c->ev_slot_free[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < EV_COUNT; ++i) CUB(cudaEventCreate(&c->ev[i]));
#undef CUB
    *out_ctx = c;
    return FYX_OK;
}

static void fyx_comm_destroy_internal(fyx_ctx *c); // fyx_comm.inl
namespace { void inst_free(fyx_ctx *c); }              // fyx_drawprep.inl
static bool lod_active(const fyx_ctx *c, uint32_t nf);  // fyx_drawprep.inl
static int32_t lod_pass(fyx_ctx *c);                    // fyx_drawprep.inl
// DFS-pruning features (LOD filter, static batches): the cull cannot be fused into the level kernels
static bool unfused_cull(const fyx_ctx *c, uint32_t nf);
static int32_t cull_unfused(fyx_ctx *c, uint32_t nf);
namespace { void anim_free(fyx_ctx *c); }              // fyx_anim.inl
static int32_t animate_enqueue(fyx_ctx *c, float dt);  // fyx_anim.inl
static int32_t allgather_enqueue(fyx_ctx *c, VisSlot &V, cudaStream_t s);
static int32_t allgather_finish(fyx_ctx *c, VisSlot &V, cudaStream_t s);
static int32_t hostseg_publish(fyx_ctx *c, VisSlot &V, cudaStream_t s);
static int32_t resolve_counts(fyx_ctx *c, VisSlot &V);

extern "C" void fyx_destroy(fyx_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    fyx_comm_destroy_internal(c);
    inst_free(c);
    anim_free(c);
    DevBuf *bufs[] = {&c->b_vis, &c->b_parent, &c->b_flags, &c->b_mask, &c->b_gidx, &c->b_slot_of_node, &c->d_stage, &c->b_statics, &c->b_trs, &c->b_vblk,
                      &c->b_ms_range, &c->b_ms_bundle, &c->b_ms_skin, &c->b_prune, &c->b_sf_rng, &c->b_opos, &c->b_onrm, &c->b_bs, &c->b_bs_w, &c->b_tblk, &c->b_otan, &c->b_bst, &c->b_surf_of_slot, &c->b_surf_bones, &c->b_palette, &c->b_bone_slot, &c->b_tiles, &c->b_fold_node,
                      &c->b_fold_begin, &c->b_fold_bone, &c->b_fold_stale_idx, &c->b_late_slot, &c->b_stale_pos, &c->b_counts_packed, &c->b_counts_all};
    for (DevBuf *b : bufs) dev_free(*b);
    for (int i = 0; i < 3; ++i) {
        dev_free(c->b_L[i]);
        dev_free(c->b_G[i]);
        dev_free(c->b_la[i]);
        dev_free(c->b_wa[i]);
        dev_free(c->b_ib[i]);
    }
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->d2h_stream) cudaStreamSynchronize(c->d2h_stream);
    if (c->fold_stream) cudaStreamSynchronize(c->fold_stream);
    for (VisSlot &V : c->vs) {
        for (uint32_t f = 0; f < FYX_MAX_FRUSTA; ++f) {
            dev_free(V.b_vis[f]);
            if (V.h_vis[f]) cudaFreeHost(V.h_vis[f]);
            dev_free(V.b_gath_pad[f]);
            dev_free(V.b_gath[f]);
            if (V.h_gath[f]) cudaFreeHost(V.h_gath[f]);
        }
        if (V.ev_gather) cudaEventDestroy(V.ev_gather);
        if (V.ev_counts_all) cudaEventDestroy(V.ev_counts_all);
        if (V.d_counts) cudaFree(V.d_counts);
        if (V.h_counts) cudaFreeHost(V.h_counts);
        if (V.ev_cull) cudaEventDestroy(V.ev_cull);
        if (V.ev_counts) cudaEventDestroy(V.ev_counts);
        if (V.ev_done) cudaEventDestroy(V.ev_done);
    }
    for (int i = 0; i < 2; ++i) {
        dev_free(c->d_stage_frame[i]);
        if (c->ev_upload[i]) cudaEventDestroy(c->ev_upload[i]);
        if (c->ev_slot_free[i]) cudaEventDestroy(c->ev_slot_free[i]);
    }
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->d2h_stream) cudaStreamDestroy(c->d2h_stream);
    if (c->fold_stream) cudaStreamDestroy(c->fold_stream);
    if (c->ev_levels_done) cudaEventDestroy(c->ev_levels_done);
    if (c->ev_fold_done) cudaEventDestroy(c->ev_fold_done);
    for (int i = 0; i < 2; ++i) {
        if (c->ev_gath_read[i]) cudaEventDestroy(c->ev_gath_read[i]);
        if (c->ev_x0[i]) cudaEventDestroy(c->ev_x0[i]);
        if (c->ev_x1[i]) cudaEventDestroy(c->ev_x1[i]);
    }
    if (c->d_err) cudaFree(c->d_err);
    if (c->h_err) cudaFreeHost(c->h_err);
    if (c->h_counts_all) cudaFreeHost(c->h_counts_all);
    if (c->h_stage) cudaFreeHost(c->h_stage);
    for (int i = 0; i < EV_COUNT; ++i)
        if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int32_t fyx_sync(fyx_ctx *c)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    return sync_and_check(c);
}

extern "C" void *fyx_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

extern "C" void fyx_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

extern "C" uint64_t fyx_kernel_launch_count(const fyx_ctx *c) { return c ? c->launches : 0; }

// --------------------------------------------------------------------------------------------
// host-side math (tiny, per frustum).  Built with -ffp-contract=off.
// --------------------------------------------------------------------------------------------
namespace {
inline float h_dot3(const float *u, const float *v) { return (u[0] * v[0] + u[1] * v[1]) + u[2] * v[2]; }
inline void h_cross(const float *u, const float *v, float *o)
{
    o[0] = u[1] * v[2] - u[2] * v[1];
    o[1] = u[2] * v[0] - u[0] * v[2];
    o[2] = u[0] * v[1] - u[1] * v[0];
}
// Plane::from_abcd — fyrox-math/src/plane.rs:63-75
bool h_plane(float a, float b, float c_, float d, float *out)
{
    const float n[3] = {a, b, c_};
    const float len = std::sqrt(h_dot3(n, n));
    if (len == 0.0f) return false;
    const float coeff = 1.0f / len;
    out[0] = a * coeff;
    out[1] = b * coeff;
    out[2] = c_ * coeff;
    out[3] = d * coeff;
    return true;
}
// Plane::intersection_point — plane.rs:94-102
void h_isect(const float *a, const float *b, const float *c_, float *out)
{
    float bc[3], ca[3], ab[3];
    h_cross(b, c_, bc);
    const float f = -1.0f / h_dot3(a, bc);
    h_cross(c_, a, ca);
    h_cross(a, b, ab);
    for (int i = 0; i < 3; ++i) out[i] = ((bc[i] * a[3] + ca[i] * b[3]) + ab[i] * c_[3]) * f;
}
} // namespace

extern "C" int32_t fyx_frustum_from_view_projection_matrix(const float m[16], fyx_frustum *out)
{
    if (!m || !out) return FYX_ERR_INVALID_ARGUMENT;
    float(*p)[4] = out->planes; // frustum.rs:55-68; m[] is nalgebra's linear (column-major) index
    if (!h_plane(m[3] + m[0], m[7] + m[4], m[11] + m[8], m[15] + m[12], p[0])) return FYX_ERR_INVALID_ARGUMENT;
    if (!h_plane(m[3] - m[0], m[7] - m[4], m[11] - m[8], m[15] - m[12], p[1])) return FYX_ERR_INVALID_ARGUMENT;
    if (!h_plane(m[3] - m[1], m[7] - m[5], m[11] - m[9], m[15] - m[13], p[2])) return FYX_ERR_INVALID_ARGUMENT;
    if (!h_plane(m[3] + m[1], m[7] + m[5], m[11] + m[9], m[15] + m[13], p[3])) return FYX_ERR_INVALID_ARGUMENT;
    if (!h_plane(m[3] - m[2], m[7] - m[6], m[11] - m[10], m[15] - m[14], p[4])) return FYX_ERR_INVALID_ARGUMENT;
    if (!h_plane(m[3] + m[2], m[7] + m[6], m[11] + m[10], m[15] + m[14], p[5])) return FYX_ERR_INVALID_ARGUMENT;
    enum { L = 0, R = 1, T = 2, B = 3, F = 4, N = 5 }; // frustum.rs:70-79
    h_isect(p[L], p[T], p[F], out->corners[0]);
    h_isect(p[L], p[B], p[F], out->corners[1]);
    h_isect(p[R], p[B], p[F], out->corners[2]);
    h_isect(p[R], p[T], p[F], out->corners[3]);
    h_isect(p[L], p[T], p[N], out->corners[4]);
    h_isect(p[L], p[B], p[N], out->corners[5]);
    h_isect(p[R], p[B], p[N], out->corners[6]);
    h_isect(p[R], p[T], p[N], out->corners[7]);
    return FYX_OK;
}

extern "C" void fyx_frustum_default(fyx_frustum *out)
{
    // Frustum::default: new_perspective(1.0, FRAC_PI_2, 0.01, 1024.0) (frustum.rs:32-43)
    float m[16] = {0};
    const float znear = 0.01f, zfar = 1024.0f;
    const float m22 = 1.0f / std::tan(1.57079632679489661923f / 2.0f);
    m[5] = m22;
    m[0] = m22 / 1.0f;
    m[10] = (zfar + znear) / (znear - zfar);
    m[14] = zfar * znear * 2.0f / (znear - zfar);
    m[11] = -1.0f;
    fyx_frustum_from_view_projection_matrix(m, out);
}

extern "C" void fyx_mat4_mul(const float a[16], const float b[16], float out[16])
{
    float r[16];
    for (int j = 0; j < 4; ++j)
        for (int i = 0; i < 4; ++i) {
            float y = a[i] * b[j * 4];
            y = y + a[4 + i] * b[j * 4 + 1];
            y = y + a[8 + i] * b[j * 4 + 2];
            y = y + a[12 + i] * b[j * 4 + 3];
            r[j * 4 + i] = y;
        }
    memcpy(out, r, sizeof r);
}

// --------------------------------------------------------------------------------------------
// scene description
// --------------------------------------------------------------------------------------------
extern "C" int32_t fyx_set_topology(fyx_ctx *c, uint32_t capacity, uint32_t root, const uint32_t *parent, const uint32_t *flags,
                                    const uint32_t *render_mask, const float *local_aabb, const uint32_t *global_index)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (capacity && !parent) return fail(c, FYX_ERR_INVALID_ARGUMENT, "parent is NULL");
    if (capacity == FYX_NONE) return fail(c, FYX_ERR_INVALID_ARGUMENT, "capacity too large");
    CU(cudaSetDevice(c->device));
    const uint32_t def_flags = FYX_NODE_VISIBILITY | FYX_NODE_ENABLED | FYX_NODE_FRUSTUM_CULLING | FYX_NODE_CAST_SHADOWS | FYX_NODE_ALIVE;
    auto fl = [&](uint32_t i) { return flags ? (flags[i] & FYX_NODE_INPUT_MASK) : def_flags; };
    auto alive = [&](uint32_t i) { return i < capacity && (fl(i) & FYX_NODE_ALIVE); };

    // depth of every alive node (parent chains; a dead / out-of-range parent counts as "no parent",
    // like Pool::try_borrow failing in graph/mod.rs:1210)
    std::vector<int32_t> depth(capacity, -1);
    std::vector<uint32_t> path;
    uint32_t max_depth = 0;
    for (uint32_t i = 0; i < capacity; ++i) {
        if (!alive(i) || depth[i] >= 0) continue;
        path.clear();
        uint32_t n = i;
        int32_t base = -1;
        while (true) {
            if (depth[n] >= 0) { base = depth[n]; break; }
            if (depth[n] == -2) return fail(c, FYX_ERR_TOPOLOGY, "cycle in parent[] through node %u", n);
            depth[n] = -2;
            path.push_back(n);
            const uint32_t p = parent[n];
            if (p == FYX_NONE || !alive(p)) break;
            n = p;
        }
        for (size_t k = path.size(); k-- > 0;) {
            base += 1;
            depth[path[k]] = base;
            max_depth = std::max<uint32_t>(max_depth, (uint32_t)base);
        }
    }
    // counting sort by depth, stable in node index
    std::vector<uint32_t> level_off(capacity ? max_depth + 2 : 1, 0);
    uint32_t n_slots = 0;
    for (uint32_t i = 0; i < capacity; ++i)
        if (alive(i)) { level_off[depth[i] + 1]++; n_slots++; }
    for (size_t l = 1; l < level_off.size(); ++l) level_off[l] += level_off[l - 1];
    std::vector<uint32_t> cursor(level_off.begin(), level_off.end());
    std::vector<uint32_t> slot_of_node(capacity, FYX_NONE), node_of_slot(n_slots);
    for (uint32_t i = 0; i < capacity; ++i)
        if (alive(i)) {
            const uint32_t s = cursor[depth[i]]++;
            slot_of_node[i] = s;
            node_of_slot[s] = i;
        }
    // within a level, order by parent slot (counting sort, stable in node index): siblings become
    // contiguous, so a warp's gather of parent rows touches one or two parents instead of 32
    {
        std::vector<uint32_t> tmp, cnt;
        for (size_t d = 1; d + 1 < level_off.size(); ++d) {
            const uint32_t plo = level_off[d - 1], phi = level_off[d], lo = level_off[d], hi = level_off[d + 1];
            if (hi - lo < 2) continue;
            cnt.assign((size_t)(phi - plo) + 1, 0);
            for (uint32_t s = lo; s < hi; ++s) cnt[slot_of_node[parent[node_of_slot[s]]] - plo + 1]++;
            for (size_t k = 1; k < cnt.size(); ++k) cnt[k] += cnt[k - 1];
            tmp.resize(hi - lo);
            for (uint32_t s = lo; s < hi; ++s) {
                const uint32_t i = node_of_slot[s];
                tmp[cnt[slot_of_node[parent[i]] - plo]++] = i;
            }
            for (uint32_t k = 0; k < hi - lo; ++k) {
                node_of_slot[lo + k] = tmp[k];
                slot_of_node[tmp[k]] = lo + k;
            }
        }
    }

    // slot-ordered host columns
    std::vector<uint32_t> h_parent(n_slots), h_flags(n_slots), h_mask(n_slots), h_gidx(n_slots);
    std::vector<float2> h_la[3];
    for (auto &v : h_la) v.resize(n_slots);
    uint32_t n_renderable = 0;
    bool any_static = false;
    for (uint32_t s = 0; s < n_slots; ++s) {
        const uint32_t i = node_of_slot[s];
        const uint32_t p = parent[i];
        h_parent[s] = (p != FYX_NONE && alive(p)) ? slot_of_node[p] : FYX_NONE;
        uint32_t f = fl(i) | F_DIRTY_SELF;
        if (i == root) f |= F_ROOT;
        if (i < c->skinned_node.size() && c->skinned_node[i]) f |= F_SKINNED;
        h_flags[s] = f;
        n_renderable += (f & FYX_NODE_RENDERABLE) ? 1u : 0u;
        any_static |= (f & FYX_NODE_STATIC_BATCH) != 0;
        h_mask[s] = render_mask ? render_mask[i] : 0xFFFFFFFFu;
        h_gidx[s] = global_index ? global_index[i] : i;
        if (local_aabb) {
            const float *b = local_aabb + 6 * (size_t)i;
            h_la[0][s] = make_float2(b[0], b[3]);
            h_la[1][s] = make_float2(b[1], b[4]);
            h_la[2][s] = make_float2(b[2], b[5]);
        } else { // AxisAlignedBoundingBox::unit(), scene/base.rs:733-735
            h_la[0][s] = h_la[1][s] = h_la[2][s] = make_float2(-0.5f, 0.5f);
        }
    }

    // Sub-forest plan: from the first level on whose sub-trees are all small (<= kSfCap nodes) and numerous relative to the
    // level's width (skeletons under a wide level of meshes), whole sub-trees are grouped so that no level of a group has
    // more than kSfCap nodes; a group is one CTA of k_update_subforest.  Not worth it for wide deep levels (each launch is
    // busy by itself): FYX_SUBFOREST=1 forces it on, =0 off.
    std::vector<uint2> sf_rng;
    uint32_t sf_first = 0, sf_levels = 0, sf_ctas = 0;
    {
        const char *env = getenv("FYX_SUBFOREST");
        const int mode = (env && *env) ? atoi(env) : -1;
        const size_t nlev = level_off.size() ? level_off.size() - 1 : 0;
        if (mode != 0 && nlev >= 4 && n_slots) {
            std::vector<uint32_t> size(n_slots, 1u);
            for (uint32_t s2 = n_slots; s2-- > 0;)
                if (h_parent[s2] != FYX_NONE) size[h_parent[s2]] += size[s2];
            // widest level at or below l: a wide level keeps a launch of its own busy, only narrow ones are launch-bound
            std::vector<uint32_t> widest(nlev + 1, 0u);
            for (size_t l = nlev; l-- > 0;) widest[l] = std::max(widest[l + 1], level_off[l + 1] - level_off[l]);
            size_t pick = 0;
            for (size_t l = 1; l + 3 <= nlev; ++l) {
                uint32_t mx = 0;
                for (uint32_t s2 = level_off[l]; s2 < level_off[l + 1]; ++s2) mx = std::max(mx, size[s2]);
                const uint64_t cnt = level_off[l + 1] - level_off[l], deep = n_slots - level_off[l];
                if (cnt && mx <= kSfCap && deep >= 8 * cnt && (mode == 1 || widest[l] <= 131072u)) { pick = l; break; }
            }
            // measured (profiles/README.md): C3 (levels of 10 k - 360 k nodes) 0.0787 -> 0.0751 ms for the stage and nothing for the
            // frame; C4 (up to 6.8 M per level) much slower.  On by default only where every deep level is narrow.
            if (pick) {
                sf_first = (uint32_t)pick;
                sf_levels = (uint32_t)(nlev - pick);
                // per level, where each sub-tree's nodes start: the sub-trees of level `pick` in slot order own consecutive ranges
                const uint32_t n_tiles = level_off[pick + 1] - level_off[pick];
                std::vector<uint32_t> tile_of(n_slots - level_off[pick]);
                std::vector<uint32_t> cnt((size_t)n_tiles * sf_levels, 0u);
                for (uint32_t s2 = level_off[pick]; s2 < n_slots; ++s2) {
                    const uint32_t rel = s2 - level_off[pick];
                    tile_of[rel] = (s2 < level_off[pick + 1]) ? rel : tile_of[h_parent[s2] - level_off[pick]];
                }
                for (size_t l = pick; l < nlev; ++l)
                    for (uint32_t s2 = level_off[l]; s2 < level_off[l + 1]; ++s2) cnt[(size_t)tile_of[s2 - level_off[pick]] * sf_levels + (l - pick)]++;
                std::vector<uint32_t> cursor(sf_levels), acc(sf_levels, 0u);
                for (uint32_t li = 0; li < sf_levels; ++li) cursor[li] = level_off[pick + li];
                auto close_group = [&]() {
                    for (uint32_t li = 0; li < sf_levels; ++li) {
                        sf_rng.push_back(make_uint2(cursor[li], cursor[li] + acc[li]));
                        cursor[li] += acc[li];
                        acc[li] = 0;
                    }
                    sf_ctas++;
                };
                for (uint32_t t = 0; t < n_tiles; ++t) {
                    bool fits = true;
                    for (uint32_t li = 0; li < sf_levels; ++li)
                        if (acc[li] + cnt[(size_t)t * sf_levels + li] > kSfCap) fits = false;
                    if (!fits) close_group();
                    for (uint32_t li = 0; li < sf_levels; ++li) acc[li] += cnt[(size_t)t * sf_levels + li];
                }
                close_group();
            }
        }
    }

    // Per-node data that is NOT an argument of this call survives it: local matrices, TRS records, transform statics,
    // bundle ids and LOD ranges of every node that was alive before and still is are carried from their old slot to the
    // new one on the device (nodes that were not alive start from the defaults).  old_of_new[s] = the old slot.
    const bool carry = c->have_topology && c->n_slots > 0 && n_slots > 0;
    DevBuf b_map;
    int32_t rc;
    if (carry) {
        std::vector<uint32_t> old_of_new(n_slots, FYX_NONE);
        for (uint32_t s2 = 0; s2 < n_slots; ++s2) {
            const uint32_t i = node_of_slot[s2];
            if (i < c->n_nodes && c->slot_of_node[i] != FYX_NONE) old_of_new[s2] = c->slot_of_node[i];
        }
        if ((rc = dev_ensure(c, b_map, (size_t)n_slots * 4))) return rc;
        CU(cudaStreamSynchronize(c->stream));
        CU(cudaMemcpy(b_map.p, old_of_new.data(), (size_t)n_slots * 4, cudaMemcpyHostToDevice));
    }
    // move one per-slot column (records of `words` u32) into a fresh allocation in the new slot order
    auto carry_column = [&](DevBuf &col, uint32_t words, const PermuteDefault &def) -> int32_t {
        DevBuf fresh;
        int32_t r2 = dev_ensure(c, fresh, std::max<size_t>(n_slots, 1) * words * 4);
        if (r2) return r2;
        launch_permute_words(c->stream, fresh.p, col.p, b_map.as<uint32_t>(), n_slots, words, def);
        c->launches++;
        cudaError_t e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) {
            dev_free(fresh);
            return fail(c, FYX_ERR_CUDA, "carrying a column over the topology change failed: %s", cudaGetErrorString(e));
        }
        dev_free(col);
        col = fresh;
        return FYX_OK;
    };
    auto f2u = [](float v) { uint32_t u; memcpy(&u, &v, 4); return u; };

    // device columns
    const size_t n = std::max<uint32_t>(n_slots, 1);
    if (carry) {
        for (int k = 0; k < 3; ++k) { // identity rows for the new nodes
            PermuteDefault d{};
            d.w[k] = f2u(1.0f);
            if ((rc = carry_column(c->b_L[k], 4, d))) return rc;
        }
        if (c->have_trs) {
            PermuteDefault d{};
            d.w[6] = d.w[7] = d.w[8] = d.w[9] = f2u(1.0f); // rotation w, scale
            if ((rc = carry_column(c->b_trs, sizeof(fyx_trs) / 4, d))) return rc;
        }
        if (c->have_statics) {
            PermuteDefault d{};
            d.w[3] = f2u(1.0f);                               // pre_rotation w
            d.w[4] = d.w[8] = d.w[12] = f2u(1.0f);            // post_rotation_matrix = identity
            if ((rc = carry_column(c->b_statics, sizeof(fyx_transform_statics) / 4, d))) return rc;
        }
        if (c->have_bundles) {
            PermuteDefault d{};
            if ((rc = carry_column(c->b_bundle, 1, d))) return rc;
        }
        if (c->have_lod) {
            PermuteDefault d{};
            d.w[0] = 0x7FC00000u; // begin = NaN: not a LOD object
            if ((rc = carry_column(c->b_lod_range, 2, d))) return rc;
        }
        dev_free(b_map);
    }
    if ((rc = dev_ensure(c, c->b_parent, n * 4))) return rc;
    if ((rc = dev_ensure(c, c->b_flags, n * 4))) return rc;
    if ((rc = dev_ensure(c, c->b_mask, n * 4))) return rc;
    if ((rc = dev_ensure(c, c->b_gidx, n * 4))) return rc;
    if ((rc = dev_ensure(c, c->b_vis, (n + 15) & ~size_t(7)))) return rc;
    CU(cudaMemset(c->b_vis.p, 0, c->b_vis.bytes));
    if ((rc = dev_ensure(c, c->b_slot_of_node, std::max<size_t>(capacity, 1) * 4))) return rc;
    for (int k = 0; k < 3; ++k) {
        if ((rc = dev_ensure(c, c->b_L[k], n * sizeof(float4)))) return rc;
        if ((rc = dev_ensure(c, c->b_G[k], n * sizeof(float4)))) return rc;
        if ((rc = dev_ensure(c, c->b_la[k], n * sizeof(float2)))) return rc;
        if ((rc = dev_ensure(c, c->b_wa[k], n * sizeof(float2)))) return rc;
    }
    CU(cudaStreamSynchronize(c->stream));
    if (n_slots) {
        CU(cudaMemcpy(c->b_parent.p, h_parent.data(), n_slots * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->b_flags.p, h_flags.data(), n_slots * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->b_mask.p, h_mask.data(), n_slots * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->b_gidx.p, h_gidx.data(), n_slots * 4, cudaMemcpyHostToDevice));
        // global matrices start as identity rows (so do the local ones of a first topology); world boxes as AABB::default()
        std::vector<float4> rows(n_slots);
        const float4 idr[3] = {make_float4(1, 0, 0, 0), make_float4(0, 1, 0, 0), make_float4(0, 0, 1, 0)};
        for (int k = 0; k < 3; ++k) {
            std::fill(rows.begin(), rows.end(), idr[k]);
            if (!carry) CU(cudaMemcpy(c->b_L[k].p, rows.data(), n_slots * sizeof(float4), cudaMemcpyHostToDevice));
            CU(cudaMemcpy(c->b_G[k].p, rows.data(), n_slots * sizeof(float4), cudaMemcpyHostToDevice));
            CU(cudaMemcpy(c->b_la[k].p, h_la[k].data(), n_slots * sizeof(float2), cudaMemcpyHostToDevice));
        }
        std::vector<float2> wdef(n_slots, make_float2(3.402823466e38f, -3.402823466e38f));
        for (int k = 0; k < 3; ++k) CU(cudaMemcpy(c->b_wa[k].p, wdef.data(), n_slots * sizeof(float2), cudaMemcpyHostToDevice));
    }
    if (capacity) CU(cudaMemcpy(c->b_slot_of_node.p, slot_of_node.data(), (size_t)capacity * 4, cudaMemcpyHostToDevice));

    const bool same_capacity = c->have_topology && capacity == c->n_nodes;
    c->n_nodes = capacity;
    c->n_slots = n_slots;
    c->root = root;
    c->n_renderable = n_renderable;
    c->maybe_static_batch = any_static;
    c->sf = SubforestPlan{};
    if (sf_ctas) {
        if ((rc = dev_ensure(c, c->b_sf_rng, sf_rng.size() * sizeof(uint2)))) return rc;
        CU(cudaMemcpy(c->b_sf_rng.p, sf_rng.data(), sf_rng.size() * sizeof(uint2), cudaMemcpyHostToDevice));
        c->sf.n_ctas = sf_ctas;
        c->sf.n_levels = sf_levels;
        c->sf.first_level = sf_first;
        c->sf.rng = c->b_sf_rng.as<uint2>();
    }
    c->slot_of_node.swap(slot_of_node);
    c->node_of_slot.swap(node_of_slot);
    c->level_off.swap(level_off);
    c->have_topology = true;
    c->updated_once = false;
    if (!carry) { // nothing to carry over (first topology, or one side empty): per-slot side tables start afresh
        c->have_statics = false;
        c->have_lod = false;
        c->have_bundles = false;
        c->n_bundle_ids = 1;
        c->have_trs = false;
    }
    if (!same_capacity) c->dfs_rank.clear(); // indexed by node: stays valid while the pool capacity does
    c->rank_on_device = false; // re-derived from dfs_rank in the new slot order
    c->ms_dirty = c->have_ms;  // the per-slot surface table too (the CSR itself is by node)
    if (c->ms_of_node.size() < capacity) c->ms_of_node.resize(capacity, make_uint2(0u, 0u));
    c->anim_csr_dirty = true; // animated nodes are addressed by slot
    c->tables_dirty = true; // bone slots depend on the slot order
    rebuild_node_arrays(c);
    return FYX_OK;
}

extern "C" int32_t fyx_set_dfs_order(fyx_ctx *c, uint32_t capacity, const uint32_t *preorder_rank)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (preorder_rank && capacity != c->n_nodes) return fail(c, FYX_ERR_INVALID_ARGUMENT, "capacity %u != topology capacity %u", capacity, c->n_nodes);
    if (preorder_rank) c->dfs_rank.assign(preorder_rank, preorder_rank + capacity);
    else c->dfs_rank.clear();
    c->rank_on_device = false;
    c->tables_dirty = true;
    return FYX_OK;
}

extern "C" int32_t fyx_set_local_matrices(fyx_ctx *c, uint32_t count, const uint32_t *idx, const float *m16)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (!count) return FYX_OK;
    if (!m16) return fail(c, FYX_ERR_INVALID_ARGUMENT, "m16 is NULL");
    CU(cudaSetDevice(c->device));
    void *d_m = nullptr, *d_i = nullptr;
    int32_t rc = stage_to_device(c, m16, (size_t)count * 64, idx, idx ? (size_t)count * 4 : 0, false, &d_m, &d_i);
    if (rc) return rc;
    launch_scatter_locals(c->stream, c->a, count, static_cast<const uint32_t *>(d_i), static_cast<const float *>(d_m),
                          c->b_slot_of_node.as<uint32_t>(), c->n_nodes, c->d_err);
    c->launches++;
    CU(cudaGetLastError());
    return FYX_OK;
}

static int32_t ensure_trs_store(fyx_ctx *c)
{
    if (c->have_trs) return FYX_OK;
    int32_t rc = dev_ensure(c, c->b_trs, std::max<size_t>(c->n_slots, 1) * sizeof(fyx_trs));
    if (rc) return rc;
    launch_fill_identity_trs(c->stream, c->b_trs.as<fyx_trs>(), c->n_slots);
    c->launches++;
    c->have_trs = true;
    return FYX_OK;
}

extern "C" int32_t fyx_set_local_rotations(fyx_ctx *c, uint32_t count, const uint32_t *idx, const float *quat_ijkw)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (!count) return FYX_OK;
    if (!quat_ijkw) return fail(c, FYX_ERR_INVALID_ARGUMENT, "rotations are NULL");
    CU(cudaSetDevice(c->device));
    int32_t rc = ensure_trs_store(c);
    if (rc) return rc;
    void *d_q = nullptr, *d_i = nullptr;
    rc = stage_to_device(c, quat_ijkw, (size_t)count * 16, idx, idx ? (size_t)count * 4 : 0, false, &d_q, &d_i);
    if (rc) return rc;
    launch_scatter_trs(c->stream, c->a, count, static_cast<const uint32_t *>(d_i), d_q, true, c->b_trs.as<fyx_trs>(),
                       c->have_statics ? c->b_statics.as<fyx_transform_statics>() : nullptr, c->b_slot_of_node.as<uint32_t>(), c->n_nodes,
                       c->d_err);
    c->launches++;
    CU(cudaGetLastError());
    return FYX_OK;
}

extern "C" int32_t fyx_set_local_trs(fyx_ctx *c, uint32_t count, const uint32_t *idx, const fyx_trs *trs)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (!count) return FYX_OK;
    if (!trs) return fail(c, FYX_ERR_INVALID_ARGUMENT, "trs is NULL");
    CU(cudaSetDevice(c->device));
    int32_t rc = ensure_trs_store(c);
    if (rc) return rc;
    void *d_t = nullptr, *d_i = nullptr;
    rc = stage_to_device(c, trs, (size_t)count * sizeof(fyx_trs), idx, idx ? (size_t)count * 4 : 0, false, &d_t, &d_i);
    if (rc) return rc;
    launch_scatter_trs(c->stream, c->a, count, static_cast<const uint32_t *>(d_i), d_t, false, c->b_trs.as<fyx_trs>(),
                       c->have_statics ? c->b_statics.as<fyx_transform_statics>() : nullptr, c->b_slot_of_node.as<uint32_t>(), c->n_nodes,
                       c->d_err);
    c->launches++;
    CU(cudaGetLastError());
    return FYX_OK;
}

extern "C" int32_t fyx_set_transform_statics(fyx_ctx *c, uint32_t count, const uint32_t *idx, const fyx_transform_statics *statics)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (!count) return FYX_OK;
    if (!statics) return fail(c, FYX_ERR_INVALID_ARGUMENT, "statics is NULL");
    CU(cudaSetDevice(c->device));
    int32_t rc;
    if (!c->have_statics) {
        if ((rc = dev_ensure(c, c->b_statics, std::max<size_t>(c->n_slots, 1) * sizeof(fyx_transform_statics)))) return rc;
        launch_fill_default_statics(c->stream, c->b_statics.as<fyx_transform_statics>(), c->n_slots);
        c->launches++;
        c->have_statics = true;
    }
    void *d_s = nullptr, *d_i = nullptr;
    rc = stage_to_device(c, statics, (size_t)count * sizeof(fyx_transform_statics), idx, idx ? (size_t)count * 4 : 0, false, &d_s, &d_i);
    if (rc) return rc;
    launch_scatter_statics(c->stream, c->a, count, static_cast<const uint32_t *>(d_i), static_cast<const fyx_transform_statics *>(d_s),
                           c->b_statics.as<fyx_transform_statics>(), c->b_slot_of_node.as<uint32_t>(), c->n_nodes);
    c->launches++;
    CU(cudaGetLastError());
    return FYX_OK;
}

static int32_t set_u32_column(fyx_ctx *c, uint32_t count, const uint32_t *idx, const uint32_t *val, int mode)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (!count) return FYX_OK;
    if (!val) return fail(c, FYX_ERR_INVALID_ARGUMENT, "values are NULL");
    CU(cudaSetDevice(c->device));
    void *d_v = nullptr, *d_i = nullptr;
    int32_t rc = stage_to_device(c, val, (size_t)count * 4, idx, idx ? (size_t)count * 4 : 0, false, &d_v, &d_i);
    if (rc) return rc;
    launch_scatter_u32(c->stream, mode == 0 ? c->a.flags : c->a.mask, count, static_cast<const uint32_t *>(d_i),
                       static_cast<const uint32_t *>(d_v), c->b_slot_of_node.as<uint32_t>(), c->n_nodes, mode);
    c->launches++;
    CU(cudaGetLastError());
    return FYX_OK;
}

extern "C" int32_t fyx_set_flags(fyx_ctx *c, uint32_t count, const uint32_t *idx, const uint32_t *flags)
{
    if (c && flags)
        for (uint32_t i = 0; i < count; ++i)
            if (flags[i] & FYX_NODE_STATIC_BATCH) c->maybe_static_batch = true; // conservative: stays on until the next topology
    return set_u32_column(c, count, idx, flags, 0);
}

extern "C" int32_t fyx_set_render_masks(fyx_ctx *c, uint32_t count, const uint32_t *idx, const uint32_t *mask)
{
    return set_u32_column(c, count, idx, mask, 1);
}

extern "C" int32_t fyx_set_local_aabbs(fyx_ctx *c, uint32_t count, const uint32_t *idx, const float *aabb)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (!count) return FYX_OK;
    if (!aabb) return fail(c, FYX_ERR_INVALID_ARGUMENT, "aabb is NULL");
    CU(cudaSetDevice(c->device));
    void *d_v = nullptr, *d_i = nullptr;
    int32_t rc = stage_to_device(c, aabb, (size_t)count * 24, idx, idx ? (size_t)count * 4 : 0, false, &d_v, &d_i);
    if (rc) return rc;
    launch_scatter_aabbs(c->stream, c->a, count, static_cast<const uint32_t *>(d_i), static_cast<const float *>(d_v),
                         c->b_slot_of_node.as<uint32_t>(), c->n_nodes);
    c->launches++;
    CU(cudaGetLastError());
    return FYX_OK;
}

// --------------------------------------------------------------------------------------------
// skinned surfaces
// --------------------------------------------------------------------------------------------
namespace {

int32_t grow_vertex_streams(fyx_ctx *c, uint64_t need)
{
    if (need <= c->vert_cap) return FYX_OK;
    int32_t rc;
    const uint64_t blocks = (need + 127) / 128 + 1; // 128-vertex blocks of 11 x 512 B
    if ((rc = dev_ensure(c, c->b_vblk, blocks * kVblkStride * sizeof(float4), true))) return rc;
    if ((rc = dev_ensure(c, c->b_opos, need * 12, true))) return rc;
    if ((rc = dev_ensure(c, c->b_onrm, need * 12, true))) return rc;
    c->vert_cap = std::min<uint64_t>({(c->b_vblk.bytes / (kVblkStride * sizeof(float4)) - 1) * 128, c->b_opos.bytes / 12, c->b_onrm.bytes / 12});
    return FYX_OK;
}

int32_t grow_bone_tables(fyx_ctx *c, uint32_t need)
{
    if (need <= c->entry_cap) return FYX_OK;
    int32_t rc;
    for (int k = 0; k < 3; ++k)
        if ((rc = dev_ensure(c, c->b_ib[k], (size_t)need * 16, true))) return rc;
    if ((rc = dev_ensure(c, c->b_palette, (size_t)need * 64, true))) return rc;
    c->entry_cap = (uint32_t)std::min<size_t>({c->b_ib[0].bytes / 16, c->b_ib[1].bytes / 16, c->b_ib[2].bytes / 16, c->b_palette.bytes / 64});
    return FYX_OK;
}

void rebuild_skin_arrays(fyx_ctx *c)
{
    SkinArrays &sk = c->sk;
    sk.n_entries = c->n_entries;
    sk.bone_slot = c->b_bone_slot.as<uint32_t>();
    for (int k = 0; k < 3; ++k) sk.ib[k] = c->b_ib[k].as<float4>();
    sk.palette = c->b_palette.as<float>();
    sk.vblk = c->b_vblk.as<float4>();
    sk.opos = c->b_opos.as<float>();
    sk.onrm = c->b_onrm.as<float>();
    sk.bs = c->b_bs.as<uint2>();
    sk.bs_w = c->b_bs_w.as<float>();
    sk.tblk = c->b_tblk.as<float4>();
    sk.otan = c->b_otan.as<float>();
    sk.bst = c->b_bst.as<uint2>();
}

constexpr uint32_t kTileQuads = 2048; // up to 8192 vertices per tile (a 5k-vertex surface is one tile)

// (re)build bone-slot, fold and tile tables from the host-side surface list
int32_t commit_surfaces(fyx_ctx *c)
{
    if (!c->tables_dirty) return FYX_OK;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    const size_t ns = c->surfaces.size();
    std::vector<uint32_t> bone_slot(c->n_entries);
    std::vector<SkinTile> tiles;
    // per skinned node: bones of all its surfaces in surface order
    std::vector<uint32_t> fold_node, fold_begin, fold_bone;
    std::vector<int64_t> fold_of_node; // node → index in fold_node, built in first-surface order
    std::vector<std::vector<uint32_t>> per_node_bones, per_node_bone_nodes;
    std::vector<uint32_t> fold_mesh_node;
    fold_of_node.assign(c->n_nodes, -1);
    for (size_t s = 0; s < ns; ++s) {
        const Surface &sf = c->surfaces[s];
        for (uint32_t b = 0; b < sf.n_bones; ++b) {
            const uint32_t bn = sf.bones[b];
            bone_slot[sf.bone_off + b] = (bn < c->n_nodes) ? c->slot_of_node[bn] : FYX_NONE;
        }
        if (sf.n_verts) {
            const uint32_t quads = (sf.n_verts + 3) / 4;
            const uint32_t nt = (quads + kTileQuads - 1) / kTileQuads;
            const uint32_t per = (quads + nt - 1) / nt;
            for (uint32_t t = 0; t < nt; ++t) {
                SkinTile tl{};
                tl.bone_off = sf.bone_off;
                tl.n_bones = sf.n_bones;
                tl.quad_start = (uint32_t)(sf.vert_off / 4 + (uint64_t)t * per);
                tl.n_quads = std::min(per, quads - t * per);
                tl.n_shapes = sf.n_shapes;
                tl.bs_off = (uint32_t)sf.bs_off;
                tl.bs_blocks = sf.bs_blocks;
                tl.w_off = sf.w_off;
                tl.local_quad0 = t * per;
                tl.tan_blk = sf.tangents ? sf.tan_blk : FYX_NONE;
                tl.tan_quad0 = sf.tan_quad0;
                tl.bst_off = sf.bst_off;
                tiles.push_back(tl);
            }
        }
        if (sf.n_bones && sf.mesh_node < c->n_nodes && c->slot_of_node[sf.mesh_node] != FYX_NONE) {
            int64_t &fi = fold_of_node[sf.mesh_node];
            if (fi < 0) {
                fi = (int64_t)per_node_bones.size();
                per_node_bones.emplace_back();
                per_node_bone_nodes.emplace_back();
                fold_node.push_back(c->slot_of_node[sf.mesh_node]);
                fold_mesh_node.push_back(sf.mesh_node);
            }
            for (uint32_t b = 0; b < sf.n_bones; ++b) {
                per_node_bones[fi].push_back(bone_slot[sf.bone_off + b]);
                per_node_bone_nodes[fi].push_back(sf.bones[b]);
            }
        }
    }
    fold_begin.push_back(0);
    // bones visited after their mesh by the reference's DFS (needs fyx_set_dfs_order) keep their pre-update position
    std::vector<uint32_t> stale_idx, late_slot;
    const bool have_rank = c->dfs_rank.size() == c->n_nodes && c->n_nodes > 0;
    for (size_t m = 0; m < per_node_bones.size(); ++m) {
        const auto &v = per_node_bones[m];
        for (size_t k = 0; k < v.size(); ++k) {
            uint32_t si = FYX_NONE;
            const uint32_t bn = per_node_bone_nodes[m][k];
            if (have_rank && v[k] != FYX_NONE && c->dfs_rank[bn] > c->dfs_rank[fold_mesh_node[m]]) {
                si = (uint32_t)late_slot.size();
                late_slot.push_back(v[k]);
            }
            stale_idx.push_back(si);
        }
        fold_bone.insert(fold_bone.end(), v.begin(), v.end());
        fold_begin.push_back((uint32_t)fold_bone.size());
    }
    int32_t rc;
    if ((rc = dev_ensure(c, c->b_bone_slot, std::max<size_t>(bone_slot.size(), 1) * 4))) return rc;
    if ((rc = dev_ensure(c, c->b_tiles, std::max<size_t>(tiles.size(), 1) * sizeof(SkinTile)))) return rc;
    if ((rc = dev_ensure(c, c->b_fold_node, std::max<size_t>(fold_node.size(), 1) * 4))) return rc;
    if ((rc = dev_ensure(c, c->b_fold_begin, fold_begin.size() * 4))) return rc;
    if ((rc = dev_ensure(c, c->b_fold_bone, std::max<size_t>(fold_bone.size(), 1) * 4))) return rc;
    CU(cudaStreamSynchronize(c->stream));
    if (!bone_slot.empty()) CU(cudaMemcpy(c->b_bone_slot.p, bone_slot.data(), bone_slot.size() * 4, cudaMemcpyHostToDevice));
    if (!tiles.empty()) CU(cudaMemcpy(c->b_tiles.p, tiles.data(), tiles.size() * sizeof(SkinTile), cudaMemcpyHostToDevice));
    if (!fold_node.empty()) CU(cudaMemcpy(c->b_fold_node.p, fold_node.data(), fold_node.size() * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->b_fold_begin.p, fold_begin.data(), fold_begin.size() * 4, cudaMemcpyHostToDevice));
    if (!fold_bone.empty()) CU(cudaMemcpy(c->b_fold_bone.p, fold_bone.data(), fold_bone.size() * 4, cudaMemcpyHostToDevice));
    {   // node -> its first skinned surface, surface -> its palette range (fyx_pack_bone_matrices)
        std::vector<uint32_t> surf_of_slot(std::max<uint32_t>(c->n_slots, 1), FYX_NONE);
        std::vector<uint2> surf_bones(std::max<size_t>(ns, 1));
        for (size_t si = 0; si < ns; ++si) {
            const Surface &sf = c->surfaces[si];
            surf_bones[si] = make_uint2(sf.bone_off, sf.n_bones);
            if (!sf.n_bones || sf.mesh_node >= c->n_nodes) continue;
            const uint32_t sl = c->slot_of_node[sf.mesh_node];
            if (sl != FYX_NONE && surf_of_slot[sl] == FYX_NONE) surf_of_slot[sl] = (uint32_t)si;
        }
        if ((rc = dev_ensure(c, c->b_surf_of_slot, surf_of_slot.size() * 4))) return rc;
        if ((rc = dev_ensure(c, c->b_surf_bones, surf_bones.size() * sizeof(uint2)))) return rc;
        CU(cudaMemcpy(c->b_surf_of_slot.p, surf_of_slot.data(), surf_of_slot.size() * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->b_surf_bones.p, surf_bones.data(), surf_bones.size() * sizeof(uint2), cudaMemcpyHostToDevice));
    }
    c->n_tiles = (uint32_t)tiles.size();
    c->any_blend_shapes = false;
    for (const Surface &sf : c->surfaces) c->any_blend_shapes |= sf.n_shapes != 0 && sf.n_verts != 0;
    c->any_tangents = false;
    for (const Surface &sf : c->surfaces) c->any_tangents |= sf.tangents && sf.n_verts != 0;
    c->max_bones = 0;
    for (const Surface &sf : c->surfaces)
        if (sf.n_verts) c->max_bones = std::max(c->max_bones, sf.n_bones);
    c->fold.n = (uint32_t)fold_node.size();
    c->fold.node_slot = c->b_fold_node.as<uint32_t>();
    c->fold.bone_begin = c->b_fold_begin.as<uint32_t>();
    c->fold.bone_slot = c->b_fold_bone.as<uint32_t>();
    c->n_late = (uint32_t)late_slot.size();
    c->fold.stale_idx = nullptr;
    c->fold.stale_pos = nullptr;
    if (c->n_late) {
        if ((rc = dev_ensure(c, c->b_fold_stale_idx, stale_idx.size() * 4))) return rc;
        if ((rc = dev_ensure(c, c->b_late_slot, late_slot.size() * 4))) return rc;
        if ((rc = dev_ensure(c, c->b_stale_pos, late_slot.size() * sizeof(float4)))) return rc;
        CU(cudaMemcpy(c->b_fold_stale_idx.p, stale_idx.data(), stale_idx.size() * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->b_late_slot.p, late_slot.data(), late_slot.size() * 4, cudaMemcpyHostToDevice));
        c->fold.stale_idx = c->b_fold_stale_idx.as<uint32_t>();
        c->fold.stale_pos = c->b_stale_pos.as<float4>();
    }
    rebuild_skin_arrays(c);
    c->tables_dirty = false;
    return FYX_OK;
}

} // namespace

extern "C" int32_t fyx_add_skinned_surface(fyx_ctx *c, uint32_t mesh_node, uint32_t n_bones, const uint32_t *bone_nodes,
                                           const float *inv_bind, uint32_t n_verts, const void *verts,
                                           const fyx_vertex_layout *layout, uint32_t *out_id)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (n_bones > FYX_MAX_BONES) return fail(c, FYX_ERR_INVALID_ARGUMENT, "n_bones %u > %u", n_bones, FYX_MAX_BONES);
    if (n_bones && (!bone_nodes || !inv_bind)) return fail(c, FYX_ERR_INVALID_ARGUMENT, "bone arrays are NULL");
    if (n_verts && (!verts || !layout)) return fail(c, FYX_ERR_INVALID_ARGUMENT, "verts/layout are NULL");
    if (n_verts && !n_bones) return fail(c, FYX_ERR_INVALID_ARGUMENT, "a skinned surface needs at least one bone");
    if (n_verts) {
        const fyx_vertex_layout &l = *layout;
        if (l.stride % 4 || l.position_offset % 4 || l.normal_offset % 4 || l.bone_weights_offset % 4 || l.bone_indices_offset % 4)
            return fail(c, FYX_ERR_UNSUPPORTED, "vertex stride and attribute offsets must be multiples of 4");
        if (l.position_offset + 12 > l.stride || l.normal_offset + 12 > l.stride || l.bone_weights_offset + 16 > l.stride ||
            l.bone_indices_offset + 4 > l.stride)
            return fail(c, FYX_ERR_INVALID_ARGUMENT, "vertex attribute outside the vertex");
    }
    CU(cudaSetDevice(c->device));
    Surface sf;
    sf.mesh_node = mesh_node;
    sf.n_bones = n_bones;
    sf.bone_off = c->n_entries;
    sf.n_verts = n_verts;
    sf.vert_off = c->n_verts_total;
    sf.bones.assign(bone_nodes, bone_nodes + n_bones);
    int32_t rc;
    if ((rc = grow_bone_tables(c, c->n_entries + n_bones))) return rc;
    const uint64_t padded = ((uint64_t)n_verts + 3) & ~uint64_t(3);
    if ((rc = grow_vertex_streams(c, c->n_verts_total + padded))) return rc;
    rebuild_skin_arrays(c);
    if (n_bones) {
        void *d_m = nullptr;
        if ((rc = stage_to_device(c, inv_bind, (size_t)n_bones * 64, nullptr, 0, false, &d_m, nullptr))) return rc;
        launch_ib_rows(c->stream, n_bones, static_cast<const float *>(d_m), c->b_ib[0].as<float4>() + sf.bone_off,
                       c->b_ib[1].as<float4>() + sf.bone_off, c->b_ib[2].as<float4>() + sf.bone_off, c->d_err);
        c->launches++;
    }
    if (n_verts) {
        void *d_v = nullptr;
        if ((rc = stage_to_device(c, verts, (size_t)n_verts * layout->stride, nullptr, 0, false, &d_v, nullptr))) return rc;
        launch_deinterleave(c->stream, n_verts, static_cast<const unsigned char *>(d_v), *layout, n_bones,
                            c->b_vblk.as<float4>(), sf.vert_off, c->d_err);
        c->launches++;
    }
    CU(cudaGetLastError());
    c->n_entries += n_bones;
    c->n_verts_total += padded;
    if (n_bones && mesh_node < c->n_nodes) {
        if (c->skinned_node.size() < c->n_nodes) c->skinned_node.resize(c->n_nodes, 0);
        if (!c->skinned_node[mesh_node]) {
            c->skinned_node[mesh_node] = 1;
            const uint32_t slot = c->slot_of_node[mesh_node];
            if (slot != FYX_NONE) {
                launch_or_u32(c->stream, c->a.flags + slot, F_SKINNED | F_DIRTY_SELF);
                c->launches++;
            }
        }
    }
    if (out_id) *out_id = (uint32_t)c->surfaces.size();
    c->surfaces.push_back(std::move(sf));
    c->tables_dirty = true;
    return FYX_OK;
}

// N4: blend shapes of a surface (BlendShapesContainer, scene/mesh/surface.rs:92-218) and their weights (Mesh::blend_shapes,
// scene/mesh/mod.rs:449-456; the renderer passes weight / 100, :794-798)
extern "C" int32_t fyx_set_blend_shapes(fyx_ctx *c, uint32_t sid, uint32_t n_shapes, const void *records, uint32_t layer_stride, const float *weights)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (sid >= c->surfaces.size()) return fail(c, FYX_ERR_INVALID_ARGUMENT, "surface id %u out of range", sid);
    if (n_shapes > FYX_MAX_BLEND_SHAPES) return fail(c, FYX_ERR_INVALID_ARGUMENT, "n_shapes %u > %u", n_shapes, FYX_MAX_BLEND_SHAPES);
    Surface &sf = c->surfaces[sid];
    if (n_shapes && !records) return fail(c, FYX_ERR_INVALID_ARGUMENT, "records are NULL");
    if (n_shapes && layer_stride < sf.n_verts) return fail(c, FYX_ERR_INVALID_ARGUMENT, "layer_stride %u < the surface's %u vertices", layer_stride, sf.n_verts);
    CU(cudaSetDevice(c->device));
    c->tables_dirty = true;
    if (!n_shapes || !sf.n_verts) {
        sf.n_shapes = 0;
        return FYX_OK;
    }
    const uint32_t bs_blocks = (sf.n_verts + 127u) / 128u;
    const uint64_t need = (uint64_t)n_shapes * bs_blocks;
    if (need > 0xFFFFFFFFull) return fail(c, FYX_ERR_INVALID_ARGUMENT, "too much blend-shape data");
    int32_t rc;
    if (need > sf.bs_cap) { // a new region at the end (an earlier, smaller region of this surface is abandoned)
        if (c->bs_used + need > 0xFFFFFFFFull) return fail(c, FYX_ERR_OUT_OF_MEMORY, "blend-shape storage exhausted");
        if ((rc = dev_ensure(c, c->b_bs, (c->bs_used + need) * kBsBlockU2 * sizeof(uint2), true))) return rc;
        sf.bs_off = c->bs_used;
        sf.bs_cap = (uint32_t)need;
        c->bs_used += need;
    }
    if (n_shapes > sf.w_cap) {
        if ((rc = dev_ensure(c, c->b_bs_w, (size_t)(c->bs_w_used + n_shapes) * sizeof(float), true))) return rc;
        sf.w_off = c->bs_w_used;
        sf.w_cap = n_shapes;
        c->bs_w_used += n_shapes;
    }
    if (sf.tangents && need > sf.bst_cap) { // the same for the tangent offsets of a tangent surface
        if (c->bst_used + need > 0xFFFFFFFFull) return fail(c, FYX_ERR_OUT_OF_MEMORY, "blend-shape storage exhausted");
        if ((rc = dev_ensure(c, c->b_bst, (c->bst_used + need) * kBstBlockU2 * sizeof(uint2), true))) return rc;
        sf.bst_off = (uint32_t)c->bst_used;
        sf.bst_cap = (uint32_t)need;
        c->bst_used += need;
    }
    sf.n_shapes = n_shapes;
    sf.bs_blocks = bs_blocks;
    rebuild_skin_arrays(c);
    std::vector<float> w(n_shapes);
    for (uint32_t i = 0; i < n_shapes; ++i) w[i] = (weights ? weights[i] : 100.0f) / 100.0f; // bs.weight / 100.0 (mesh/mod.rs:797)
    void *d_rec = nullptr, *d_w = nullptr;
    if ((rc = stage_to_device(c, records, (size_t)n_shapes * layer_stride * 18, w.data(), (size_t)n_shapes * 4, false, &d_rec, &d_w))) return rc;
    launch_bs_layout(c->stream, sf.n_verts, n_shapes, layer_stride, static_cast<const uint16_t *>(d_rec), c->b_bs.as<uint2>() + sf.bs_off * kBsBlockU2, bs_blocks);
    c->launches++;
    if (sf.tangents) {
        launch_bs_tan_layout(c->stream, sf.n_verts, n_shapes, layer_stride, static_cast<const uint16_t *>(d_rec),
                             c->b_bst.as<uint2>() + (size_t)sf.bst_off * kBstBlockU2, bs_blocks);
        c->launches++;
    }
    CU(cudaMemcpyAsync(c->b_bs_w.as<float>() + sf.w_off, d_w, (size_t)n_shapes * 4, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream)); // `w` and the staging buffer are free again
    return FYX_OK;
}

// Skinned tangents of a surface (standard.shader:197-200): its VertexBuffer bytes again, tangent = f32 x4 at tangent_offset
extern "C" int32_t fyx_set_skinned_tangents(fyx_ctx *c, uint32_t sid, const void *verts, uint32_t stride, uint32_t tangent_offset)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (sid >= c->surfaces.size()) return fail(c, FYX_ERR_INVALID_ARGUMENT, "surface id %u out of range", sid);
    Surface &sf = c->surfaces[sid];
    if (!verts) {
        if (sf.tangents) c->tables_dirty = true;
        sf.tangents = false;
        return FYX_OK;
    }
    if (stride % 4 || tangent_offset % 4) return fail(c, FYX_ERR_INVALID_ARGUMENT, "vertex stride and tangent offset must be multiples of 4");
    if ((uint64_t)tangent_offset + 16 > stride) return fail(c, FYX_ERR_INVALID_ARGUMENT, "tangent (16 B at %u) outside the %u-byte vertex", tangent_offset, stride);
    if (sf.n_shapes)
        return fail(c, FYX_ERR_STATE, "surface %u already has blend shapes: call fyx_set_skinned_tangents before fyx_set_blend_shapes", sid);
    CU(cudaSetDevice(c->device));
    int32_t rc;
    const uint64_t quads = ((uint64_t)sf.n_verts + 3) / 4, blocks = (quads + 31) / 32;
    if (sf.tan_blk == FYX_NONE && sf.n_verts) { // the surface's regions, kept for the rest of its life
        if (c->tan_blocks_used + blocks > 0xFFFFFFFFull || c->tan_quads_used + quads > 0xFFFFFFFFull)
            return fail(c, FYX_ERR_OUT_OF_MEMORY, "tangent storage exhausted");
        if ((rc = dev_ensure(c, c->b_tblk, (c->tan_blocks_used + blocks) * kTblkStride * sizeof(float4), true))) return rc;
        if ((rc = dev_ensure(c, c->b_otan, (c->tan_quads_used + quads) * 48, true))) return rc;
        sf.tan_blk = (uint32_t)c->tan_blocks_used;
        sf.tan_quad0 = (uint32_t)c->tan_quads_used;
        c->tan_blocks_used += blocks;
        c->tan_quads_used += quads;
        rebuild_skin_arrays(c);
    }
    if (sf.n_verts) {
        void *d_v = nullptr;
        if ((rc = stage_to_device(c, verts, (size_t)sf.n_verts * stride, nullptr, 0, false, &d_v, nullptr))) return rc;
        launch_tan_deinterleave(c->stream, sf.n_verts, static_cast<const unsigned char *>(d_v), stride, tangent_offset,
                                c->b_tblk.as<float4>() + (size_t)sf.tan_blk * kTblkStride);
        c->launches++;
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(c->stream)); // the staging buffer is free again
    }
    sf.tangents = true;
    c->tables_dirty = true;
    return FYX_OK;
}

extern "C" int32_t fyx_set_blend_shape_weights(fyx_ctx *c, uint32_t sid, uint32_t n, const float *weights)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (sid >= c->surfaces.size()) return fail(c, FYX_ERR_INVALID_ARGUMENT, "surface id %u out of range", sid);
    Surface &sf = c->surfaces[sid];
    if (n != sf.n_shapes) return fail(c, FYX_ERR_INVALID_ARGUMENT, "the surface has %u blend shapes, %u weights given", sf.n_shapes, n);
    if (!n) return FYX_OK;
    if (!weights) return fail(c, FYX_ERR_INVALID_ARGUMENT, "weights are NULL");
    CU(cudaSetDevice(c->device));
    std::vector<float> w(n);
    for (uint32_t i = 0; i < n; ++i) w[i] = weights[i] / 100.0f;
    void *d_w = nullptr;
    int32_t rc = stage_to_device(c, w.data(), (size_t)n * 4, nullptr, 0, false, &d_w, nullptr);
    if (rc) return rc;
    CU(cudaMemcpyAsync(c->b_bs_w.as<float>() + sf.w_off, d_w, (size_t)n * 4, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return FYX_OK;
}

extern "C" int32_t fyx_reserve_skinning(fyx_ctx *c, uint64_t total_bones, uint64_t total_verts)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (total_bones > 0xFFFFFFFFull) return fail(c, FYX_ERR_INVALID_ARGUMENT, "too many bones");
    CU(cudaSetDevice(c->device));
    int32_t rc = grow_bone_tables(c, (uint32_t)total_bones);
    if (rc) return rc;
    // every surface is padded to a multiple of 4 vertices: leave room for 3 per surface (bounded by bones)
    rc = grow_vertex_streams(c, total_verts + 4 * total_bones + 4);
    if (rc) return rc;
    rebuild_skin_arrays(c);
    return FYX_OK;
}

extern "C" int32_t fyx_commit_surfaces(fyx_ctx *c)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    CU(cudaSetDevice(c->device));
    int32_t rc = commit_surfaces(c);
    if (rc) return rc;
    return sync_and_check(c);
}

// --------------------------------------------------------------------------------------------
// per frame
// --------------------------------------------------------------------------------------------
extern "C" int32_t fyx_update_transforms(fyx_ctx *c, uint32_t update_flags)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    CU(cudaSetDevice(c->device));
    int32_t rc = commit_surfaces(c);
    if (rc) return rc;
    CU(cudaEventRecord(c->ev[EV_START], c->stream));
    rc = run_update(c, update_flags, nullptr);
    if (rc) return rc;
    CU(cudaEventRecord(c->ev[EV_UPDATE], c->stream));
    rc = sync_and_check(c);
    cudaEventElapsedTime(&c->timings.update_ms, c->ev[EV_START], c->ev[EV_UPDATE]);
    return rc;
}

extern "C" int32_t fyx_cull(fyx_ctx *c, uint32_t nf, const fyx_frustum *fr, const uint32_t *cam_mask, const uint32_t *pass_flags)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    CU(cudaSetDevice(c->device));
    CU(cudaEventRecord(c->ev[EV_START], c->stream));
    int32_t rc = prepare_cull(c, nf, fr, cam_mask, pass_flags);
    if (rc) return rc;
    if (nf && (rc = cull_unfused(c, nf))) return rc;
    CU(cudaEventRecord(c->ev[EV_CULL], c->stream));
    rc = sync_and_check(c);
    cudaEventElapsedTime(&c->timings.cull_ms, c->ev[EV_START], c->ev[EV_CULL]);
    return rc;
}

extern "C" int32_t fyx_update_and_cull(fyx_ctx *c, uint32_t update_flags, uint32_t nf, const fyx_frustum *fr,
                                       const uint32_t *cam_mask, const uint32_t *pass_flags)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    CU(cudaSetDevice(c->device));
    int32_t rc = commit_surfaces(c);
    if (rc) return rc;
    CU(cudaEventRecord(c->ev[EV_START], c->stream));
    rc = prepare_cull(c, nf, fr, cam_mask, pass_flags);
    if (rc) return rc;
    {
        // with a LOD filter / static batches the cull cannot be fused into the level kernels: the pruning bits need every ancestor first
        const bool unf = unfused_cull(c, nf);
        rc = run_update(c, update_flags, (nf && !unf) ? &c->cp : nullptr);
        if (rc) return rc;
        if (unf && (rc = cull_unfused(c, nf))) return rc;
    }
    CU(cudaEventRecord(c->ev[EV_UPDATE], c->stream));
    rc = sync_and_check(c);
    cudaEventElapsedTime(&c->timings.update_ms, c->ev[EV_START], c->ev[EV_UPDATE]);
    return rc;
}

extern "C" int32_t fyx_get_visible(fyx_ctx *c, uint32_t f, const uint32_t **out_idx, uint32_t *out_count)
{
    if (!c || !out_idx || !out_count) return FYX_ERR_INVALID_ARGUMENT;
    VisSlot &V = c->vs[c->readable];
    if (V.pending) return fail(c, FYX_ERR_STATE, "the frame is still in flight: call fyx_frame_wait first");
    if (f >= V.nf) return fail(c, FYX_ERR_INVALID_ARGUMENT, "frustum %u was not part of the last cull (%u frusta)", f, V.nf);
    CU(cudaSetDevice(c->device));
    int32_t rc = readback_visible(c, V, c->stream);
    if (rc) return rc;
    *out_idx = V.own_in_seg ? V.seg_own[f] : V.h_vis[f]; // a gathered frame's own lists sit inside the node-wide host segment
    *out_count = V.h_counts[f];
    return FYX_OK;
}

extern "C" int32_t fyx_get_visible_device(fyx_ctx *c, uint32_t f, const uint32_t **d_idx, const uint32_t **d_count)
{
    if (!c || !d_idx || !d_count) return FYX_ERR_INVALID_ARGUMENT;
    VisSlot &V = c->vs[c->cur];
    if (f >= V.nf) return fail(c, FYX_ERR_INVALID_ARGUMENT, "frustum %u was not part of the last cull (%u frusta)", f, V.nf);
    *d_idx = V.b_vis[f].as<uint32_t>();
    *d_count = V.d_counts + f * kCountStride;
    return FYX_OK;
}

extern "C" int32_t fyx_build_palettes(fyx_ctx *c)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    CU(cudaSetDevice(c->device));
    int32_t rc = commit_surfaces(c);
    if (rc) return rc;
    CU(cudaEventRecord(c->ev[EV_START], c->stream));
    if (c->sk.n_entries) {
        launch_palette(c->stream, c->a, c->sk);
        c->launches++;
    }
    CU(cudaEventRecord(c->ev[EV_PALETTE], c->stream));
    rc = sync_and_check(c);
    cudaEventElapsedTime(&c->timings.palette_ms, c->ev[EV_START], c->ev[EV_PALETTE]);
    return rc;
}

extern "C" int32_t fyx_skin(fyx_ctx *c)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    CU(cudaSetDevice(c->device));
    int32_t rc = commit_surfaces(c);
    if (rc) return rc;
    CU(cudaEventRecord(c->ev[EV_START], c->stream));
    if (c->n_tiles) {
        launch_skin(c->stream, c->sk, c->b_tiles.as<SkinTile>(), c->n_tiles, c->max_bones, c->any_blend_shapes, c->any_tangents);
        c->launches++;
    }
    CU(cudaEventRecord(c->ev[EV_SKIN], c->stream));
    rc = sync_and_check(c);
    cudaEventElapsedTime(&c->timings.skin_ms, c->ev[EV_START], c->ev[EV_SKIN]);
    return rc;
}

static void frame_timings_from_events(fyx_ctx *c)
{
    fyx_timings &t = c->timings;
    t.upload_ms = t.update_ms = t.palette_ms = t.skin_ms = t.readback_ms = 0.0f;
    if (c->stage_events_valid) {
        cudaEventElapsedTime(&t.upload_ms, c->ev[EV_START], c->ev[EV_UPLOAD]);
        cudaEventElapsedTime(&t.update_ms, c->ev[EV_UPLOAD], c->ev[EV_UPDATE]);
        cudaEventElapsedTime(&t.palette_ms, c->ev[EV_UPDATE], c->ev[EV_PALETTE]);
        cudaEventElapsedTime(&t.skin_ms, c->ev[EV_PALETTE], c->ev[EV_SKIN]);
        cudaEventElapsedTime(&t.readback_ms, c->ev[EV_SKIN], c->ev[EV_READBACK]);
    }
    cudaEventElapsedTime(&t.total_ms, c->ev[EV_START], c->ev[EV_READBACK]);
    t.cull_ms = 0.0f;
    c->timings_pending = false;
}

extern "C" int32_t fyx_render_prep(fyx_ctx *c, const fyx_frame_desc *fr)
{
    if (!c || !fr) return FYX_ERR_INVALID_ARGUMENT;
    if (fr->struct_size < offsetof(fyx_frame_desc, do_animate)) return fail(c, FYX_ERR_INVALID_ARGUMENT, "fyx_frame_desc.struct_size too small");
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    CU(cudaSetDevice(c->device));
    int32_t rc = commit_surfaces(c);
    if (rc) return rc;
    cudaStream_t s = c->stream;
    CU(cudaEventRecord(c->ev[EV_START], s));
    // 0. animation players tick before Graph::update (N2): curves are device-resident, nothing to upload
    if (fr->struct_size >= sizeof(fyx_frame_desc) && fr->do_animate) {
        rc = animate_enqueue(c, fr->animate_dt);
        if (rc) return rc;
    }
    const bool async = (fr->flags & FYX_FRAME_ASYNC) != 0;
    // Per-stage events sit BETWEEN kernels of the programmatic-dependent-launch chain and would keep a kernel's
    // prologue from overlapping its predecessor's tail: only synchronous frames record them (their timings are read
    // right after the call); asynchronous frames record the frame's start and end only (stage fields read 0).
    const bool stage_events = !async;
    c->stage_events_valid = stage_events;
    const bool pipelined = async && fr->readback_visible && fr->n_frusta; // read-back deferred to fyx_frame_wait
    bool side_fold = false;
    // 1. changed local matrices.  Pinned caller memory is DMA'd in place (the caller keeps it untouched until
    //    the frame is synchronised / waited for).  Async frames upload on the copy stream into alternating
    //    staging buffers, so the H2D of frame i+1 overlaps the kernels of frame i.
    if (fr->n_changed) {
        const bool as_rot = fr->changed_rot != nullptr, as_trs = !as_rot && fr->changed_trs != nullptr;
        const void *payload = as_rot ? static_cast<const void *>(fr->changed_rot)
                                     : (as_trs ? static_cast<const void *>(fr->changed_trs) : static_cast<const void *>(fr->changed_m16));
        if (!payload) return fail(c, FYX_ERR_INVALID_ARGUMENT, "changed_m16 / changed_trs / changed_rot is NULL");
        if (as_rot || as_trs) {
            rc = ensure_trs_store(c);
            if (rc) return rc;
        }
        const size_t mb = (size_t)fr->n_changed * (as_rot ? 16 : (as_trs ? sizeof(fyx_trs) : 64)), ib = fr->changed_idx ? (size_t)fr->n_changed * 4 : 0;
        const fyx_transform_statics *st = c->have_statics ? c->b_statics.as<fyx_transform_statics>() : nullptr;
        auto scatter = [&](cudaStream_t ss, const void *d_p, const uint32_t *d_i) {
            if (as_rot || as_trs)
                launch_scatter_trs(ss, c->a, fr->n_changed, d_i, d_p, as_rot, c->b_trs.as<fyx_trs>(), st, c->b_slot_of_node.as<uint32_t>(),
                                   c->n_nodes, c->d_err);
            else
                launch_scatter_locals(ss, c->a, fr->n_changed, d_i, static_cast<const float *>(d_p), c->b_slot_of_node.as<uint32_t>(),
                                      c->n_nodes, c->d_err);
        };
        if (async && is_pinned(payload) && (!fr->changed_idx || is_pinned(fr->changed_idx))) {
            const int u = (c->upload_parity ^= 1);
            if (c->slot_used[u]) CU(cudaEventSynchronize(c->ev_slot_free[u])); // its previous scatter has consumed it
            const size_t off = (mb + 255) & ~size_t(255);
            rc = dev_ensure(c, c->d_stage_frame[u], off + ib + 256);
            if (rc) return rc;
            char *base = c->d_stage_frame[u].as<char>();
            CU(cudaMemcpyAsync(base, payload, mb, cudaMemcpyHostToDevice, c->copy_stream));
            if (ib) CU(cudaMemcpyAsync(base + off, fr->changed_idx, ib, cudaMemcpyHostToDevice, c->copy_stream));
            // The scatter writes local matrices / TRS records / F_DIRTY_SELF of the changed nodes — columns nothing of the PREVIOUS
            // frame reads once its level kernels and fold are done.  When that point is known (the previous frame recorded its
            // cull event) and nothing else has been enqueued on the main stream since, the scatter runs on the copy stream, beside
            // the previous frame's palette / skinning kernels, instead of in front of this frame's level kernels.
            static const bool side_allowed = [] {
                const char *e = getenv("FYX_SIDE_SCATTER"); // 0: always scatter on the main stream (A/B measurements)
                return !(e && *e == '0');
            }();
            const bool side = side_allowed && c->ev_levels_prev && c->launches == c->launches_at_frame_end &&
                              !(fr->struct_size >= sizeof(fyx_frame_desc) && fr->do_animate);
            if (side) {
                CU(cudaStreamWaitEvent(c->copy_stream, c->ev_levels_prev, 0));
                scatter(c->copy_stream, base, ib ? reinterpret_cast<const uint32_t *>(base + off) : nullptr);
                CU(cudaEventRecord(c->ev_upload[u], c->copy_stream));
                CU(cudaEventRecord(c->ev_slot_free[u], c->copy_stream));
                CU(cudaStreamWaitEvent(s, c->ev_upload[u], 0));
            } else {
                CU(cudaEventRecord(c->ev_upload[u], c->copy_stream));
                CU(cudaStreamWaitEvent(s, c->ev_upload[u], 0));
                scatter(s, base, ib ? reinterpret_cast<const uint32_t *>(base + off) : nullptr);
                CU(cudaEventRecord(c->ev_slot_free[u], s));
            }
            c->slot_used[u] = true;
        } else {
            void *d_m = nullptr, *d_i = nullptr;
            rc = stage_to_device(c, payload, mb, fr->changed_idx, ib, true, &d_m, &d_i);
            if (rc) return rc;
            scatter(s, d_m, static_cast<const uint32_t *>(d_i));
        }
        c->launches++;
    }
    if (stage_events) CU(cudaEventRecord(c->ev[EV_UPLOAD], s));
    // 2. hierarchy + world boxes + cull
    if (fr->n_frusta) {
        rc = prepare_cull(c, fr->n_frusta, fr->frusta, fr->cam_mask, fr->pass_flags);
        if (rc) return rc;
    }
    {
        const bool unf = unfused_cull(c, fr->n_frusta);
        static const bool side_fold_allowed = [] {
            const char *e = getenv("FYX_SIDE_FOLD"); // 0: the fold always runs in order on the main stream (A/B measurements)
            return !(e && *e == '0');
        }();
        side_fold = side_fold_allowed && async && !unf && c->fold.n && fr->do_skin && c->n_tiles;
        rc = run_update(c, fr->update_flags, (fr->n_frusta && !unf) ? &c->cp : nullptr, side_fold ? c->fold_stream : nullptr);
        if (rc) return rc;
        if (unf && (rc = cull_unfused(c, fr->n_frusta))) return rc;
    }
    if (stage_events) CU(cudaEventRecord(c->ev[EV_UPDATE], s));
    c->ev_levels_prev = nullptr;
    if (fr->n_frusta && (async || (fr->flags & FYX_FRAME_ALLGATHER))) {
        // consumed by the read-back / collective streams and by the next frame's scatter: the lists are complete after the fold
        CU(cudaEventRecord(c->vs[c->cur].ev_cull, side_fold ? c->fold_stream : s));
        c->ev_levels_prev = c->vs[c->cur].ev_cull;
    }
    // multi-GPU: the visible lists are complete here; their all-gather runs on the collective stream beside
    // the palette / skinning kernels below (the path's one exchange step, SURVEY §8e)
    const bool gather = (fr->flags & FYX_FRAME_ALLGATHER) && fr->n_frusta;
    if (gather) {
        if (!c->comm) return fail(c, FYX_ERR_STATE, "FYX_FRAME_ALLGATHER without fyx_comm_init");
        CU(cudaStreamWaitEvent(c->comm_stream, c->vs[c->cur].ev_cull, 0));
        if (c->vs[c->cur ^ 1].gathered) CU(cudaStreamWaitEvent(c->comm_stream, c->vs[c->cur ^ 1].ev_gather, 0)); // a stand-alone exchange of the previous frame
        c->vs[c->cur].host_copy_private = !fr->readback_visible; // nobody promised that every rank fetches this frame's lists
        rc = allgather_enqueue(c, c->vs[c->cur], c->comm_stream);
        if (rc) return rc;
    }
    // 3. palettes, 4. skinning
    if (fr->do_palettes && c->sk.n_entries) {
        launch_palette(s, c->a, c->sk);
        c->launches++;
    }
    if (stage_events) CU(cudaEventRecord(c->ev[EV_PALETTE], s));
    if (fr->do_skin && c->n_tiles) {
        launch_skin(s, c->sk, c->b_tiles.as<SkinTile>(), c->n_tiles, c->max_bones, c->any_blend_shapes, c->any_tangents);
        c->launches++;
    }
    if (stage_events) CU(cudaEventRecord(c->ev[EV_SKIN], s));
    CU(cudaGetLastError());
    if (side_fold) CU(cudaStreamWaitEvent(s, c->ev_fold_done, 0)); // join: whatever follows on the main stream sees the folded boxes and the complete lists
    if (gather) {
        // the host waits only for the cull + the counts (the skinning kernel keeps running), then enqueues the payload
        rc = allgather_finish(c, c->vs[c->cur], c->comm_stream);
        if (rc) return rc;
        CU(cudaEventRecord(c->ev_x1[c->vs[c->cur].epoch & 1], c->comm_stream));
        CU(cudaEventRecord(c->vs[c->cur].ev_gather, c->comm_stream));
        CU(cudaStreamWaitEvent(s, c->vs[c->cur].ev_gather, 0)); // the frame is complete when the gathered lists are
    }
    // 5. visible lists to the host
    VisSlot &V = c->vs[c->cur];
    if (pipelined) {
        // deferred: counts travel on the read-back stream as soon as the cull is done; fyx_frame_wait fetches the lists
        CU(cudaEventRecord(V.ev_done, s));
        CU(cudaStreamWaitEvent(c->d2h_stream, V.ev_cull, 0));
        CU(cudaMemcpy2DAsync(V.h_counts, sizeof(uint32_t), V.d_counts, sizeof(uint32_t) * kCountStride, sizeof(uint32_t), V.nf,
                             cudaMemcpyDeviceToHost, c->d2h_stream));
        CU(cudaEventRecord(V.ev_counts, c->d2h_stream));
        V.pending = true;
        V.own_only = gather && (fr->flags & FYX_FRAME_READBACK_OWN);
        V.frame_no = ++c->frame_counter;
    } else if (fr->readback_visible && fr->n_frusta && !gather) {
        rc = readback_visible(c, V, s);
        if (rc) return rc;
    } // with FYX_FRAME_ALLGATHER the frame's result is the gathered lists: fyx_get_visible_gathered fetches them
    CU(cudaEventRecord(c->ev[EV_READBACK], s));
    c->launches_at_frame_end = c->launches;
    if (async) {
        c->timings_pending = true;
        return FYX_OK;
    }
    rc = sync_and_check(c);
    frame_timings_from_events(c);
    if (!rc && gather && fr->readback_visible && c->hostseg_ready) rc = hostseg_publish(c, V, s); // every rank's part, without being asked
    return rc;
}

// Collect the oldest pipelined frame: wait for its kernels, bring its visible lists to the host, make it
// the frame fyx_get_visible reads.  No-op when nothing is in flight.
extern "C" int32_t fyx_frame_wait(fyx_ctx *c)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    int slot = -1;
    for (int i = 0; i < 2; ++i)
        if (c->vs[i].pending && (slot < 0 || c->vs[i].frame_no < c->vs[slot].frame_no)) slot = i;
    if (slot < 0) return FYX_OK;
    CU(cudaSetDevice(c->device));
    VisSlot &V = c->vs[slot];
    CU(cudaEventSynchronize(V.ev_counts));
    V.counts_on_host = true;
    const bool seg = V.gathered && c->hostseg_ready && !V.host_copy_private;
    const bool own = !seg && (!V.gathered || V.own_only);
    for (uint32_t f = 0; f < V.nf && own; ++f) {
        const size_t n = V.h_counts[f];
        int32_t rc = host_list_ensure(c, V, f, n);
        if (rc) return rc;
        if (n) CU(cudaMemcpyAsync(V.h_vis[f], V.b_vis[f].p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->d2h_stream));
    }
    if (seg) {
        // multi-GPU frame: this rank's own lists go into the node-wide host segment at their offsets (every rank does the
        // same over its own PCIe link); fyx_get_visible_gathered reads the whole lists there
        int32_t rc = hostseg_publish(c, V, c->d2h_stream);
        if (rc) return rc;
    } else if (V.gathered && !V.own_only) { // no segment: the host wants the whole (all-gathered) lists from this rank's device
        int32_t rc = resolve_counts(c, V);
        if (rc) return rc;
        CU(cudaStreamWaitEvent(c->d2h_stream, V.ev_gather, 0));
        for (uint32_t f = 0; f < V.nf; ++f) {
            const size_t n = V.gath_count[f];
            rc = host_gath_ensure(c, V, f, n);
            if (rc) return rc;
            if (n) CU(cudaMemcpyAsync(V.h_gath[f], V.gath_ptr[f], n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->d2h_stream));
        }
        CU(cudaEventRecord(c->ev_gath_read[V.epoch & 1], c->d2h_stream));
        c->gath_read_valid[V.epoch & 1] = true;
        V.gathered_on_host = true;
    }
    CU(cudaStreamWaitEvent(c->d2h_stream, V.ev_done, 0)); // the error word is final once the frame's last kernel ran
    CU(cudaMemcpyAsync(c->h_err, c->d_err, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->d2h_stream));
    CU(cudaStreamSynchronize(c->d2h_stream));
    V.lists_on_host = own || V.own_in_seg;
    V.pending = false;
    c->readable = slot;
    return check_device_errors(c);
}

// --------------------------------------------------------------------------------------------
// read-back
// --------------------------------------------------------------------------------------------
namespace {
// gather `count` items of `item_bytes` through a gather launcher into caller memory
template <class Launch> int32_t gather_out(fyx_ctx *c, uint32_t count, const uint32_t *idx, size_t item_bytes, void *out, Launch launch)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (!c->have_topology) return fail(c, FYX_ERR_STATE, "fyx_set_topology has not been called");
    if (!count) return FYX_OK;
    if (!out) return fail(c, FYX_ERR_INVALID_ARGUMENT, "output pointer is NULL");
    CU(cudaSetDevice(c->device));
    const size_t out_bytes = (size_t)count * item_bytes;
    const size_t idx_bytes = idx ? (((size_t)count * 4 + 255) & ~size_t(255)) : 0;
    int32_t rc = dev_ensure(c, c->d_stage, idx_bytes + out_bytes);
    if (rc) return rc;
    char *base = c->d_stage.as<char>();
    uint32_t *d_idx = nullptr;
    if (idx) {
        CU(cudaStreamSynchronize(c->stream));
        CU(cudaMemcpyAsync(base, idx, (size_t)count * 4, cudaMemcpyHostToDevice, c->stream));
        d_idx = reinterpret_cast<uint32_t *>(base);
    }
    launch(d_idx, base + idx_bytes);
    c->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, base + idx_bytes, out_bytes, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return FYX_OK;
}
} // namespace

extern "C" int32_t fyx_get_global_matrices(fyx_ctx *c, uint32_t count, const uint32_t *idx, float *out)
{
    return gather_out(c, count, idx, 64, out, [&](uint32_t *d_idx, void *d_out) {
        launch_gather_globals(c->stream, c->a, count, d_idx, c->b_slot_of_node.as<uint32_t>(), c->n_nodes, static_cast<float *>(d_out));
    });
}

extern "C" int32_t fyx_get_world_aabbs(fyx_ctx *c, uint32_t count, const uint32_t *idx, float *out)
{
    return gather_out(c, count, idx, 24, out, [&](uint32_t *d_idx, void *d_out) {
        launch_gather_aabbs(c->stream, c->a, count, d_idx, c->b_slot_of_node.as<uint32_t>(), c->n_nodes, static_cast<float *>(d_out));
    });
}

extern "C" int32_t fyx_get_global_flags(fyx_ctx *c, uint32_t count, const uint32_t *idx, uint32_t *out)
{
    return gather_out(c, count, idx, 4, out, [&](uint32_t *d_idx, void *d_out) {
        launch_gather_flags(c->stream, c->a, count, d_idx, c->b_slot_of_node.as<uint32_t>(), c->n_nodes, static_cast<uint32_t *>(d_out));
    });
}

extern "C" int32_t fyx_get_palette(fyx_ctx *c, uint32_t sid, float *out)
{
    if (!c || !out) return FYX_ERR_INVALID_ARGUMENT;
    if (sid >= c->surfaces.size()) return fail(c, FYX_ERR_INVALID_ARGUMENT, "surface id %u out of range", sid);
    CU(cudaSetDevice(c->device));
    const Surface &sf = c->surfaces[sid];
    if (!sf.n_bones) return FYX_OK;
    CU(cudaMemcpyAsync(out, c->b_palette.as<float>() + 16 * (size_t)sf.bone_off, (size_t)sf.n_bones * 64, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return FYX_OK;
}

extern "C" int32_t fyx_get_skinned(fyx_ctx *c, uint32_t sid, float *out_pos, float *out_nrm)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (sid >= c->surfaces.size()) return fail(c, FYX_ERR_INVALID_ARGUMENT, "surface id %u out of range", sid);
    CU(cudaSetDevice(c->device));
    const Surface &sf = c->surfaces[sid];
    if (!sf.n_verts) return FYX_OK;
    if (out_pos) CU(cudaMemcpyAsync(out_pos, c->b_opos.as<float>() + 3 * sf.vert_off, (size_t)sf.n_verts * 12, cudaMemcpyDeviceToHost, c->stream));
    if (out_nrm) CU(cudaMemcpyAsync(out_nrm, c->b_onrm.as<float>() + 3 * sf.vert_off, (size_t)sf.n_verts * 12, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return FYX_OK;
}

extern "C" int32_t fyx_get_skinned_device(fyx_ctx *c, uint32_t sid, const float **d_pos, const float **d_nrm)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (sid >= c->surfaces.size()) return fail(c, FYX_ERR_INVALID_ARGUMENT, "surface id %u out of range", sid);
    const Surface &sf = c->surfaces[sid];
    if (d_pos) *d_pos = c->b_opos.as<float>() + 3 * sf.vert_off;
    if (d_nrm) *d_nrm = c->b_onrm.as<float>() + 3 * sf.vert_off;
    return FYX_OK;
}

extern "C" int32_t fyx_get_skinned_tangents(fyx_ctx *c, uint32_t sid, float *out_tan3)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (sid >= c->surfaces.size()) return fail(c, FYX_ERR_INVALID_ARGUMENT, "surface id %u out of range", sid);
    const Surface &sf = c->surfaces[sid];
    if (!sf.tangents) return fail(c, FYX_ERR_STATE, "surface %u has no skinned tangents (fyx_set_skinned_tangents)", sid);
    if (!sf.n_verts) return FYX_OK;
    if (!out_tan3) return fail(c, FYX_ERR_INVALID_ARGUMENT, "out_tan3 is NULL");
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(out_tan3, c->b_otan.as<float>() + 12 * (size_t)sf.tan_quad0, (size_t)sf.n_verts * 12, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return FYX_OK;
}

extern "C" int32_t fyx_get_skinned_tangents_device(fyx_ctx *c, uint32_t sid, const float **d_tan3)
{
    if (!c) return FYX_ERR_INVALID_ARGUMENT;
    if (sid >= c->surfaces.size()) return fail(c, FYX_ERR_INVALID_ARGUMENT, "surface id %u out of range", sid);
    const Surface &sf = c->surfaces[sid];
    if (!sf.tangents) return fail(c, FYX_ERR_STATE, "surface %u has no skinned tangents (fyx_set_skinned_tangents)", sid);
    if (d_tan3) *d_tan3 = sf.n_verts ? c->b_otan.as<float>() + 12 * (size_t)sf.tan_quad0 : nullptr;
    return FYX_OK;
}

extern "C" int32_t fyx_get_timings(fyx_ctx *c, fyx_timings *out)
{
    if (!c || !out) return FYX_ERR_INVALID_ARGUMENT;
    if (c->timings_pending) {
        CU(cudaSetDevice(c->device));
        CU(cudaEventSynchronize(c->ev[EV_READBACK]));
        frame_timings_from_events(c);
    }
    *out = c->timings;
    return FYX_OK;
}

#include "fyx_comm.inl"
#include "fyx_drawprep.inl"
#include "fyx_anim.inl"
