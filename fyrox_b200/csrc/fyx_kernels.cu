// fyx_kernels.cu — hand-written sm_100a kernels of the render-prep hot path.
//
// All kernels are HBM-bandwidth-bound streaming kernels over SoA planes (no tensor cores: 4x4 f32
// work at ~0.3-1 flop/B).  Arithmetic follows fyx_math.cuh (one rounding per op, reference order).
// Each kernel names the reference code it replaces (paths relative to the Fyrox tree).
#include <cstdlib>
#include <cstring>

#include <cuda_fp16.h>

#include "fyx_internal.h"
#include "fyx_trs.cuh"

namespace fyx {

// ------------------------------------------------------------------------------------------------
// streaming load/store helpers: node columns are touched once per frame ⇒ bypass L1 allocation for the
// big streams (read-only path, evict-first), keep default caching for the gathered parent rows.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ld_stream(const float4 *p)
{
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ float2 ld_stream(const float2 *p)
{
    float2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_stream(const uint4 *p)
{
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream(float4 *p, const float4 v)
{
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
__device__ __forceinline__ void st_stream(float2 *p, const float2 v)
{
    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}

// ------------------------------------------------------------------------------------------------
// Programmatic dependent launch: the kernels of a frame form a chain of true data dependencies (level l
// needs level l-1, the fold needs every level, the palettes the bones, the skinning the palettes), several
// of them tiny.  Each is launched with programmatic stream serialization: it lets the next kernel's CTAs be
// scheduled right away (pdl_trigger) and waits for the previous kernel's results only where it first needs
// them (pdl_wait) — launch latency and the loads that do not depend on the predecessor overlap its tail.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <class... Params, class... Args>
static void launch_pdl(void (*kernel)(Params...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<Params>(args)...);
}

// ------------------------------------------------------------------------------------------------
// Warp-level pre-reject of whole frusta (the 6-frusta cull is instruction-issue-bound, not HBM-bound).
//
// Siblings sit in adjacent slots, so the 32 boxes of a warp are neighbours in the world and most frusta of a
// multi-frustum call (five of six cube faces, typically) contain none of them.  The warp reduces its boxes to
// their union U and tests U ONCE, with the work spread over the lanes: lane l < 3*nf evaluates plane pair
// l%3 of frustum l/3 on U's max-corner, lane c (two rounds) tests frustum corner c against U.  Frustum f is
// dead for the warp iff some plane rejects U and no corner of f lies in U; then every participating lane's
// own test is false too, bit for bit:
//   * cloud test: for a lane box B ⊆ U the operand picked per axis (min for a negative normal component, max
//     otherwise) is never further along the normal than U's, products by the same constant and sums are
//     monotone under round-to-nearest, so s_B <= s_U <= 0 on that plane — the lane's max-corner (hence all
//     eight corners, frustum.rs:205-219) is behind it;
//   * fallback (frustum.rs:236-242): a corner outside U on some axis (exact compares) is outside B on it.
// Participating lanes = candidates with frustum culling on and a tame box (finite, ordered: the premise of
// the max-corner form); everything else keeps its own per-lane test.  CPU check of the claim on random and
// adversarial warps: tests/test_cull_trick_cpu.py.
// ------------------------------------------------------------------------------------------------
struct PrefTable {
    float4 e[FYX_MAX_FRUSTA * 3][5];      // per (frustum, plane pair): pn[0..3] (2 float4), vsel[3][2] (6 u32), pad: 80 B stride = conflict-free LDS.128
    float4 corner[FYX_MAX_FRUSTA * 8];
};

__device__ __forceinline__ void pref_fill(PrefTable &T, const CullParams &cp, const int nf)
{
    const int t = threadIdx.x;
    if (t < 3 * nf) {
        const int f = t / 3, q = t % 3;
        const FrustumDev &F = cp.f[f];
        T.e[t][0] = make_float4(F.pn[q][0].x, F.pn[q][0].y, F.pn[q][1].x, F.pn[q][1].y);
        T.e[t][1] = make_float4(F.pn[q][2].x, F.pn[q][2].y, F.pn[q][3].x, F.pn[q][3].y);
        T.e[t][2] = make_float4(__uint_as_float(F.vsel[q][0][0]), __uint_as_float(F.vsel[q][0][1]), __uint_as_float(F.vsel[q][1][0]),
                                __uint_as_float(F.vsel[q][1][1]));
        T.e[t][3] = make_float4(__uint_as_float(F.vsel[q][2][0]), __uint_as_float(F.vsel[q][2][1]), 0.f, 0.f);
    }
    const int c = t - 64;
    if (c >= 0 && c < 8 * nf) T.corner[c] = cp.f[c >> 3].corner[c & 7];
}

__device__ __forceinline__ float warp_min_f32(const float v)
{
    float r;
    asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float warp_max_f32(const float v)
{
    float r;
    asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
    return r;
}

// Must be called by all 32 lanes.  part: this lane's box takes part in the union.  Returns the frusta that are NOT
// proven dead for the participating lanes (bit f).
template <int NFT>
__device__ __forceinline__ uint32_t warp_live_frusta(const bool part, const float2 wx, const float2 wy, const float2 wz, const int nf_rt,
                                                     const PrefTable &T, const PackedConsts &kc)
{
    const int nf = (NFT > 0) ? NFT : nf_rt;
    if (!__any_sync(0xFFFFFFFFu, part)) return 0u; // nobody needs a geometric test
    const float inf = __int_as_float(0x7f800000);
    const float ulx = warp_min_f32(part ? wx.x : inf), uhx = warp_max_f32(part ? wx.y : -inf);
    const float uly = warp_min_f32(part ? wy.x : inf), uhy = warp_max_f32(part ? wy.y : -inf);
    const float ulz = warp_min_f32(part ? wz.x : inf), uhz = warp_max_f32(part ? wz.y : -inf);
    const int lane = threadIdx.x & 31;
    bool rej = false;
    if (lane < 3 * nf) {
        const float4 a = T.e[lane][0], b = T.e[lane][1], s0 = T.e[lane][2], s1 = T.e[lane][3];
        const uint32_t xl = __float_as_uint(ulx), xh = __float_as_uint(uhx), yl = __float_as_uint(uly), yh = __float_as_uint(uhy),
                       zl = __float_as_uint(ulz), zh = __float_as_uint(uhz);
        const float2 vx = make_float2(pick(xl, xh, __float_as_uint(s0.x)), pick(xl, xh, __float_as_uint(s0.y)));
        const float2 vy = make_float2(pick(yl, yh, __float_as_uint(s0.z)), pick(yl, yh, __float_as_uint(s0.w)));
        const float2 vz = make_float2(pick(zl, zh, __float_as_uint(s1.x)), pick(zl, zh, __float_as_uint(s1.y)));
        const float2 s = add2(add2(add2(mul2(make_float2(a.x, a.y), vx, kc), mul2(make_float2(a.z, a.w), vy, kc), kc),
                                   mul2(make_float2(b.x, b.y), vz, kc), kc), make_float2(b.z, b.w), kc);
        rej = (s.x <= 0.0f) | (s.y <= 0.0f);
    }
    const uint32_t rb = __ballot_sync(0xFFFFFFFFu, rej);
    uint32_t live = 0u;
    constexpr int kRounds = (NFT > 0) ? (8 * NFT + 31) / 32 : (8 * (int)FYX_MAX_FRUSTA + 31) / 32;
#pragma unroll
    for (int r = 0; r < kRounds; ++r) {
        if (NFT == 0 && r * 4 >= nf) break;
        const int c = lane + 32 * r;
        bool in = false;
        if (c < 8 * nf) {
            const float4 k = T.corner[c];
            in = (k.x >= ulx) & (k.x <= uhx) & (k.y >= uly) & (k.y <= uhy) & (k.z >= ulz) & (k.z <= uhz);
        }
        const uint32_t cb = __ballot_sync(0xFFFFFFFFu, in);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int f = 4 * r + j;
            if (f < nf) {
                const bool cloud_fail = ((rb >> (3 * f)) & 7u) != 0u;
                const bool corner_in = ((cb >> (8 * j)) & 0xFFu) != 0u;
                live |= (!cloud_fail || corner_in) ? (1u << f) : 0u;
            }
        }
    }
    return live;
}

// ------------------------------------------------------------------------------------------------
// NodeTrait::should_be_rendered (scene/node/mod.rs:231-256) + the shadow-pass cast_shadows test of
// Mesh::collect_render_data (scene/mesh/mod.rs:696-698) + reachability from Graph::root
// (iterate_recursive, renderer/bundle.rs:988-1004), for every frustum of the call.  Bit f of the
// result = "node is in the visible set of frustum f".
// ------------------------------------------------------------------------------------------------
// NFT: number of frusta known at compile time (the loop is unrolled and cp.f[f] becomes constant-bank operands of the
// arithmetic instead of ~35 indexed parameter loads per frustum), 0 = run-time count.
// live: frusta whose geometric test this lane still has to run (all ones without the warp-level pre-reject).
constexpr uint32_t kNeedBits = FYX_NODE_ALIVE | FYX_NODE_RENDERABLE | FYX_NODE_REACHABLE | FYX_NODE_GLOBAL_VISIBILITY | FYX_NODE_GLOBAL_ENABLED;

template <int NFT>
__device__ __forceinline__ uint32_t cull_bits(const uint32_t nf, const uint32_t mask, const float2 wx, const float2 wy,
                                              const float2 wz, const CullParams &cp, const PackedConsts &kc, const bool tame, const uint32_t live)
{
    if ((nf & kNeedBits) != kNeedBits) return 0u;
    uint32_t bits = 0u;
    auto one = [&](const int f) {
        bool ok = (mask & cp.f[f].cam_mask) != 0u;
        ok &= !((cp.f[f].pass_flags & FYX_PASS_SHADOW) && !(nf & FYX_NODE_CAST_SHADOWS));
        if (ok && (nf & FYX_NODE_FRUSTUM_CULLING)) {
            // a frustum proven dead for the warp's union box needs no test — unless this lane's box is not tame (it took
            // no part in the union)
            if (((live >> f) & 1u) || !tame) ok = frustum_intersects_aabb(cp.f[f], wx, wy, wz, kc, tame);
            else ok = false;
        }
        bits |= ok ? (1u << f) : 0u;
    };
    if (NFT > 0) {
#pragma unroll
        for (int f = 0; f < NFT; ++f) one(f);
    } else {
        for (int f = 0; f < cp.nf; ++f) one(f);
    }
    return bits;
}

// Per-warp part of the cull, called by all 32 lanes: cand = this lane holds a node that may be emitted at all.
// PRE: warp-level pre-reject on.
template <int NFT, bool PRE>
__device__ __forceinline__ uint32_t cull_warp(const bool cand, const uint32_t nf, const uint32_t mask, const float2 wx, const float2 wy,
                                              const float2 wz, const CullParams &cp, const PrefTable *T)
{
    PackedConsts kc;
    kc.one = make_float2(cp.one, cp.one);
    kc.negzero = make_float2(cp.negzero, cp.negzero);
    const bool ok = cand && (nf & kNeedBits) == kNeedBits;
    const bool tame = ok && aabb_is_tame(wx, wy, wz);
    uint32_t live = 0xFFFFFFFFu;
    if (PRE) live = warp_live_frusta<NFT>(tame && (nf & FYX_NODE_FRUSTUM_CULLING), wx, wy, wz, cp.nf, *T, kc);
    return ok ? cull_bits<NFT>(nf, mask, wx, wy, wz, cp, kc, tame, live) : 0u;
}

// ------------------------------------------------------------------------------------------------
// The same predicate in warp-convergent form (VAR bit 5), called by all 32 lanes.  The per-lane form above runs the
// geometric test inside `if (ok && culling)`: every frustum costs a divergence region (BSSY/BSYNC, an activemask per
// vote) and ~12 instructions of mask / pass / flag tests.  Here
//   * the cheap tests produce one bit mask of eligible frusta per lane (per call: shadow passes as a bit mask, the
//     camera masks compared once when they are all equal);
//   * the plane tests of frustum f run for the WHOLE warp whenever some lane needs them (the other lanes' values are
//     ignored: same issue slots either way), so every vote uses the full mask and every branch is warp-uniform;
//   * the corner-in-box fallback runs only for lanes a plane rejected without the margin of `pm` (fyx_math.cuh).
// Lanes whose box is not tame (never in practice) take the literal per-lane test.  Same booleans as cull_bits.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool corner_in_box(const FrustumDev &f, const float2 x, const float2 y, const float2 z)
{
    uint32_t alive = 0xFFu;
    const float2 box[3] = {x, y, z};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float lo = box[a].x, hi = box[a].y;
        const float4 v0 = f.ax_val[a][0];
        uint32_t m = 0u;
        m |= ((v0.x >= lo) & (v0.x <= hi)) ? f.ax_mask[a][0] : 0u;
        m |= ((v0.y >= lo) & (v0.y <= hi)) ? f.ax_mask[a][1] : 0u;
        m |= ((v0.z >= lo) & (v0.z <= hi)) ? f.ax_mask[a][2] : 0u;
        m |= ((v0.w >= lo) & (v0.w <= hi)) ? f.ax_mask[a][3] : 0u;
        if (((f.n_ax >> (8 * a)) & 0xFFu) > 4u) {
            const float4 v1 = f.ax_val[a][1];
            m |= ((v1.x >= lo) & (v1.x <= hi)) ? f.ax_mask[a][4] : 0u;
            m |= ((v1.y >= lo) & (v1.y <= hi)) ? f.ax_mask[a][5] : 0u;
            m |= ((v1.z >= lo) & (v1.z <= hi)) ? f.ax_mask[a][6] : 0u;
            m |= ((v1.w >= lo) & (v1.w <= hi)) ? f.ax_mask[a][7] : 0u;
        }
        alive &= m;
    }
    return alive != 0u;
}

template <int NFT>
__device__ __forceinline__ uint32_t cull_warp_conv(const bool cand, const uint32_t nf, const uint32_t mask, const float2 wx, const float2 wy,
                                                   const float2 wz, const CullParams &cp)
{
    constexpr uint32_t kFull = 0xFFFFFFFFu;
    PackedConsts kc;
    kc.one = make_float2(cp.one, cp.one);
    kc.negzero = make_float2(cp.negzero, cp.negzero);
    const int nfr = (NFT > 0) ? NFT : cp.nf;
    const uint32_t all = (nfr >= 32) ? kFull : ((1u << nfr) - 1u);
    const bool ok = cand && (nf & kNeedBits) == kNeedBits;
    // eligible frusta of this lane: render mask ∩ camera mask, shadow passes only for shadow casters
    uint32_t elig;
    if (cp.cam_same) {
        elig = (mask & cp.f[0].cam_mask) ? all : 0u;
    } else {
        elig = 0u;
        if (NFT > 0) {
#pragma unroll
            for (int f = 0; f < NFT; ++f) elig |= (mask & cp.f[f].cam_mask) ? (1u << f) : 0u;
        } else {
            for (int f = 0; f < nfr; ++f) elig |= (mask & cp.f[f].cam_mask) ? (1u << f) : 0u;
        }
    }
    if (!(nf & FYX_NODE_CAST_SHADOWS)) elig &= ~cp.shadow_bits;
    if (!ok) elig = 0u;
    const bool geo = (nf & FYX_NODE_FRUSTUM_CULLING) != 0u;
    uint32_t want = geo ? elig : 0u; // frusta whose geometric test this lane needs
    if (!__any_sync(kFull, want != 0u)) return elig;
    uint32_t bits = geo ? 0u : elig;
    const bool tame = aabb_is_tame(wx, wy, wz);
    if (__any_sync(kFull, want != 0u && !tame)) { // literal per-lane path for boxes outside the max-corner form's premise
        if (want != 0u && !tame) {
            for (int f = 0; f < nfr; ++f)
                if (((want >> f) & 1u) && frustum_intersects_aabb(cp.f[f], wx, wy, wz, kc, false)) bits |= 1u << f;
            want = 0u;
        }
    }
    const uint32_t xl = __float_as_uint(wx.x), xh = __float_as_uint(wx.y), yl = __float_as_uint(wy.x), yh = __float_as_uint(wy.y),
                   zl = __float_as_uint(wz.x), zh = __float_as_uint(wz.y);
    auto one = [&](const int f) {
        const bool act = ((want >> f) & 1u) != 0u;
        if (!__any_sync(kFull, act)) return;
        const FrustumDev &F = cp.f[f];
        bool cloud = act, strong = false;
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const float2 vx = make_float2(pick(xl, xh, F.vsel[q][0][0]), pick(xl, xh, F.vsel[q][0][1]));
            const float2 vy = make_float2(pick(yl, yh, F.vsel[q][1][0]), pick(yl, yh, F.vsel[q][1][1]));
            const float2 vz = make_float2(pick(zl, zh, F.vsel[q][2][0]), pick(zl, zh, F.vsel[q][2][1]));
            const float2 s = add2(add2(add2(mul2(F.pn[q][0], vx, kc), mul2(F.pn[q][1], vy, kc), kc), mul2(F.pn[q][2], vz, kc), kc), F.pn[q][3], kc);
            cloud &= !(s.x <= 0.0f) & !(s.y <= 0.0f);
            strong |= (s.x < F.pm[q].x) | (s.y < F.pm[q].y);
            if (q < 2 && !__any_sync(kFull, cloud)) break; // every lane that wanted this frustum is rejected already
        }
        bool res = cloud;
        const bool fb = act && !cloud && !strong; // rejected by a plane it (nearly) touches: the reference's corner loop decides
        if (__any_sync(kFull, fb)) {
            if (fb) res = corner_in_box(F, wx, wy, wz);
        }
        bits |= res ? (1u << f) : 0u;
    };
    if (NFT > 0) {
#pragma unroll
        for (int f = 0; f < NFT; ++f) one(f);
    } else {
        for (int f = 0; f < nfr; ++f) one(f);
    }
    return bits;
}

// ------------------------------------------------------------------------------------------------
// Compaction of the visible node indices.  Replaces the Vec pushes of RenderDataBundleStorage::push
// (renderer/bundle.rs:1248-1278).  Order inside a list is unspecified.  Two forms:
//  * CTA-wide: warp ballot + popc rank, per-warp counts in shared memory, one atomicAdd per (CTA, frustum);
//  * warp-wide: one atomicAdd per (warp, frustum that has a visible lane) — no shared memory, no barriers, and
//    frusta nobody in the warp is visible in cost nothing (the 6-frusta kernel is issue-bound: ~180 -> ~30
//    instructions per warp); the counters sit on their own 128 B lines.
// Both must be called by every thread of the CTA / warp.
// ------------------------------------------------------------------------------------------------
template <int NFT>
__device__ __forceinline__ void compact_emit(const uint32_t vis_bits, const uint32_t node_index, const uint32_t slot,
                                             const CullParams &cp)
{
    constexpr int kWarps = kBlock / 32;
    __shared__ uint32_t s_wcount[FYX_MAX_FRUSTA][kWarps];
    __shared__ uint32_t s_base[FYX_MAX_FRUSTA];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nf = (NFT > 0) ? NFT : cp.nf;

    // any visible node in the CTA at all?  (most CTAs of a mostly-culled scene skip the atomics)
    const int any = __syncthreads_or(vis_bits != 0u);
    if (!any) return;

    for (int f = 0; f < nf; ++f) {
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, (vis_bits >> f) & 1u);
        if (lane == 0) s_wcount[f][warp] = __popc(b);
    }
    __syncthreads();
    if (threadIdx.x < nf) {
        const int f = threadIdx.x;
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const uint32_t c = s_wcount[f][w];
            s_wcount[f][w] = run; // exclusive prefix over warps
            run += c;
        }
        s_base[f] = run ? atomicAdd(cp.counts + f * kCountStride, run) : 0u;
    }
    __syncthreads();
    for (int f = 0; f < nf; ++f) {
        const uint32_t bit = (vis_bits >> f) & 1u;
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, bit);
        if (bit) {
            const uint32_t pos = s_base[f] + s_wcount[f][warp] + __popc(b & ((1u << lane) - 1u));
            cp.out[f][pos] = node_index;
            if (cp.out_slot[f]) cp.out_slot[f][pos] = slot; // where the node lives in HBM (fyx_pack_instances)
        }
    }
}

__device__ __forceinline__ void compact_emit_warp(const uint32_t vis_bits, const uint32_t node_index, const uint32_t slot, const CullParams &cp)
{
    uint32_t m = __reduce_or_sync(0xFFFFFFFFu, vis_bits); // frusta with a visible lane in this warp (uniform)
    const uint32_t lane = threadIdx.x & 31u;
    while (m) {
        const int f = __ffs(m) - 1;
        m &= m - 1u;
        const uint32_t bit = (vis_bits >> f) & 1u;
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, bit);
        uint32_t base = 0u;
        if (lane == 0) base = atomicAdd(cp.counts + f * kCountStride, (uint32_t)__popc(b));
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (bit) {
            const uint32_t pos = base + __popc(b & ((1u << lane) - 1u));
            cp.out[f][pos] = node_index;
            if (cp.out_slot[f]) cp.out_slot[f][pos] = slot;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// One hierarchy level.  Replaces, for the nodes of this level:
//   Graph::update_global_transform_recursively   scene/graph/mod.rs:1199-1241   (G = parent.G * local)
//   Graph::update_visibility_recursively          :1182-1197                      (gv = parent.gv && visibility)
//   Graph::update_enabled_flag_recursively        :1166-1180                      (ge = parent.ge && enabled)
//   Mesh::on_global_transform_changed / Base::world_bounding_box   scene/mesh/mod.rs:667-689, scene/base.rs:741-750
//   (+ (NFT >= 0): should_be_rendered + visible-list emission for non-skinned nodes)
// and the change tracking of process_node_messages (:1303-1399): a node is recomputed iff it or an
// ancestor changed (or FYX_UPDATE_ALL).  One thread per node; parents were finished by the previous
// launch on the same stream.
// Algorithmic bytes per node (SURVEY §8d): 132 (T) + 48 (A) [+ 8 (K)]; moved: 48+4+48 + 24+24 + 4+4(+4+4).
// ------------------------------------------------------------------------------------------------
// (A single cooperative launch walking all levels with grid-wide barriers was tried and rejected: the
// persistent grid, L2-only parent loads and the barriers cost more than the launches they save —
// C2 0.357 -> 0.416 ms, target 0.990 -> 1.051 ms per frame; profiles/README.md.)
// UA: FYX_UPDATE_ALL known at compile time — every load of the node's own columns is issued at once, next to the load of
// the parent index, instead of after the parent's flags have said whether the node is dirty (two dependent memory
// round trips per node instead of three; the kernel is latency-bound: ncu long_scoreboard 8 of 17 stalled warps per issue).
template <bool WANT_BOX, bool UA>
__device__ __forceinline__ void update_node(const NodeArrays &a, const uint32_t slot, const uint32_t update_all, uint32_t &nf_out, float2 &wx,
                                            float2 &wy, float2 &wz)
{
    const uint32_t p = a.parent[slot]; // static column: may be read before the predecessor has finished
    pdl_wait(); // everything below reads what the previous level / a scatter kernel / the previous frame's tail wrote
    const uint32_t f = a.flags[slot]; // mutable (F_DIRTY_SELF is set by the scatter kernels): only after the wait
    Affine L;
    float2 lx, ly, lz;
    if (UA) {
        L.r0 = ld_stream(a.L[0] + slot);
        L.r1 = ld_stream(a.L[1] + slot);
        L.r2 = ld_stream(a.L[2] + slot);
        lx = ld_stream(a.la[0] + slot);
        ly = ld_stream(a.la[1] + slot);
        lz = ld_stream(a.la[2] + slot);
    }
    // no parent ⇒ parent values are identity / true (graph/mod.rs:1171-1175,1187-1192,1210-1214)
    const uint32_t pf = (p != FYX_NONE)
                            ? a.flags[p]
                            : (FYX_NODE_GLOBAL_VISIBILITY | FYX_NODE_GLOBAL_ENABLED | ((f & F_ROOT) ? FYX_NODE_REACHABLE : 0u));
    const bool dirty = UA || update_all || (f & F_DIRTY_SELF) || (pf & F_DIRTY);
    uint32_t nf = f & ~(FYX_NODE_GLOBAL_VISIBILITY | FYX_NODE_GLOBAL_ENABLED | FYX_NODE_REACHABLE | F_DIRTY | F_DIRTY_SELF);
    if ((pf & FYX_NODE_GLOBAL_VISIBILITY) && (f & FYX_NODE_VISIBILITY)) nf |= FYX_NODE_GLOBAL_VISIBILITY;
    if ((pf & FYX_NODE_GLOBAL_ENABLED) && (f & FYX_NODE_ENABLED)) nf |= FYX_NODE_GLOBAL_ENABLED;
    nf |= pf & FYX_NODE_REACHABLE;
    if (dirty) nf |= F_DIRTY;
    a.flags[slot] = nf;
    nf_out = nf;

    if (dirty) {
        if (!UA) {
            L.r0 = ld_stream(a.L[0] + slot);
            L.r1 = ld_stream(a.L[1] + slot);
            L.r2 = ld_stream(a.L[2] + slot);
            lx = ld_stream(a.la[0] + slot);
            ly = ld_stream(a.la[1] + slot);
            lz = ld_stream(a.la[2] + slot);
        }
        Affine P;
        if (p != FYX_NONE) {
            P.r0 = a.G[0][p]; // siblings are adjacent slots: one or two parents per warp (L1 hits)
            P.r1 = a.G[1][p];
            P.r2 = a.G[2][p];
        } else {
            P = affine_identity();
        }
        const Affine Gm = affine_mul(P, L);
        st_stream(a.G[0] + slot, Gm.r0);
        st_stream(a.G[1] + slot, Gm.r1);
        st_stream(a.G[2] + slot, Gm.r2);
        wx = aabb_transform_row(Gm.r0, lx, ly, lz);
        wy = aabb_transform_row(Gm.r1, lx, ly, lz);
        wz = aabb_transform_row(Gm.r2, lx, ly, lz);
        // skinned meshes: this is the box before the bone fold; fold_mesh finishes it
        st_stream(a.wa[0] + slot, wx);
        st_stream(a.wa[1] + slot, wy);
        st_stream(a.wa[2] + slot, wz);
    } else if (WANT_BOX) {
        wx = ld_stream(a.wa[0] + slot);
        wy = ld_stream(a.wa[1] + slot);
        wz = ld_stream(a.wa[2] + slot);
    }
}

// VAR: bit 0 = warp-level pre-reject of whole frusta, bit 1 = warp-wide compaction (else CTA-wide), bit 2 = FYX_UPDATE_ALL
// specialisation (own columns, render mask and list index loaded up front)
// bit 4 = compiled for 8 resident CTAs per SM (<= 32 registers: the 40 the kernel wants limit it to 48 of 64 warps, and it is
// latency-bound); bit 5 = warp-convergent predicate (cull_warp_conv; replaces bit 0)
template <int NFT, int VAR>
__global__ void __launch_bounds__(kBlock, (VAR & 16) ? 8 : 6) k_update_level(const NodeArrays a, const uint32_t lo, const uint32_t hi,
                                                         const uint32_t update_all, const CullParams cp)
{
    pdl_trigger();
    constexpr bool PRE = (NFT >= 0) && (VAR & 1);
    constexpr bool UA = (VAR & 4) != 0;
    __shared__ __align__(16) unsigned char s_pref[PRE ? sizeof(PrefTable) : 16];
    PrefTable *T = reinterpret_cast<PrefTable *>(s_pref);
    if (PRE) {
        pref_fill(*T, cp, NFT > 0 ? NFT : cp.nf);
        __syncthreads();
    }
    const uint32_t slot = lo + blockIdx.x * kBlock + threadIdx.x;
    uint32_t nf = 0u;
    float2 wx = make_float2(0.f, 0.f), wy = wx, wz = wx;
    const bool valid = slot < hi;
    uint32_t mask = 0u, gi_early = 0u;
    if (UA && (NFT >= 0) && valid) { // static columns: no reason to wait for anything
        mask = a.mask[slot];
        if (!(VAR & 8)) gi_early = a.gidx[slot];
    }
    if (valid) update_node<(NFT >= 0), UA>(a, slot, update_all, nf, wx, wy, wz);
    else pdl_wait();
    if (NFT >= 0) {
        const bool cand = valid && !(nf & F_SKINNED);
        if (!UA) mask = cand ? a.mask[slot] : 0u;
        const uint32_t vis_bits = (VAR & 32) ? cull_warp_conv<(NFT > 0 ? NFT : 0)>(cand, nf, mask, wx, wy, wz, cp)
                                             : cull_warp<(NFT > 0 ? NFT : 0), PRE>(cand, nf, mask, wx, wy, wz, cp, T);
        if (VAR & 8) { // deferred compaction: one byte per node now, the lists are built by k_compact_vis after the last level
            if (valid) a.vis[slot] = (uint8_t)vis_bits;
            return;
        }
        const uint32_t gi = UA ? gi_early : (vis_bits ? a.gidx[slot] : 0u);
        if (VAR & 2) compact_emit_warp(vis_bits, gi, slot, cp);
        else compact_emit<(NFT > 0 ? NFT : 0)>(vis_bits, gi, slot, cp);
    }
}

// ------------------------------------------------------------------------------------------------
// The deep levels of the hierarchy in ONE launch (SubforestPlan, fyx_internal.h): a CTA owns a group of whole
// sub-trees — e.g. a dozen 64-bone skeletons — and walks their levels itself.  In every level the group's nodes are one
// contiguous slot range (coalesced like a level kernel); the matrices and flags of the previous level stay in shared
// memory for the children.  Same arithmetic, flags, change tracking and fused cull as k_update_level; what it removes
// is a kernel launch per level for levels of a few thousand nodes (C3: six skeleton levels of 10 k - 320 k nodes).
// ------------------------------------------------------------------------------------------------
template <int NFT, bool UA, bool DEFER>
__global__ void __launch_bounds__(kBlock) k_update_subforest(const NodeArrays a, const uint2 *__restrict__ rng, const int n_levels,
                                                             const uint32_t update_all, const CullParams cp)
{
    pdl_trigger();
    __shared__ float4 s_g[2][3][kSfCap];
    __shared__ uint32_t s_f[2][kSfCap];
    const uint2 *my = rng + (size_t)blockIdx.x * n_levels;
    pdl_wait();
    uint32_t prevA = 0u, prevB = 0u;
    for (int li = 0; li < n_levels; ++li) {
        const uint2 r = my[li];
        const int cur = li & 1, prv = cur ^ 1;
        for (uint32_t base = r.x; base < r.y; base += kBlock) { // the same trip count for every thread of the CTA
            const uint32_t slot = base + threadIdx.x;
            const bool valid = slot < r.y;
            uint32_t nf = 0u;
            float2 wx = make_float2(0.f, 0.f), wy = wx, wz = wx;
            if (valid) {
                const uint32_t p = a.parent[slot];
                const uint32_t f = a.flags[slot];
                Affine L;
                float2 lx, ly, lz;
                if (UA) {
                    L.r0 = ld_stream(a.L[0] + slot);
                    L.r1 = ld_stream(a.L[1] + slot);
                    L.r2 = ld_stream(a.L[2] + slot);
                    lx = ld_stream(a.la[0] + slot);
                    ly = ld_stream(a.la[1] + slot);
                    lz = ld_stream(a.la[2] + slot);
                }
                const bool in_prev = (li > 0) && (p >= prevA) && (p < prevB); // the parent was handled by this CTA one level up
                const uint32_t pf = in_prev ? s_f[prv][p - prevA]
                                            : ((p != FYX_NONE) ? a.flags[p]
                                                               : (FYX_NODE_GLOBAL_VISIBILITY | FYX_NODE_GLOBAL_ENABLED | ((f & F_ROOT) ? FYX_NODE_REACHABLE : 0u)));
                const bool dirty = UA || update_all || (f & F_DIRTY_SELF) || (pf & F_DIRTY);
                nf = f & ~(FYX_NODE_GLOBAL_VISIBILITY | FYX_NODE_GLOBAL_ENABLED | FYX_NODE_REACHABLE | F_DIRTY | F_DIRTY_SELF);
                if ((pf & FYX_NODE_GLOBAL_VISIBILITY) && (f & FYX_NODE_VISIBILITY)) nf |= FYX_NODE_GLOBAL_VISIBILITY;
                if ((pf & FYX_NODE_GLOBAL_ENABLED) && (f & FYX_NODE_ENABLED)) nf |= FYX_NODE_GLOBAL_ENABLED;
                nf |= pf & FYX_NODE_REACHABLE;
                if (dirty) nf |= F_DIRTY;
                a.flags[slot] = nf;
                const uint32_t me = slot - r.x;
                s_f[cur][me] = nf;
                Affine Gm;
                if (dirty) {
                    if (!UA) {
                        L.r0 = ld_stream(a.L[0] + slot);
                        L.r1 = ld_stream(a.L[1] + slot);
                        L.r2 = ld_stream(a.L[2] + slot);
                        lx = ld_stream(a.la[0] + slot);
                        ly = ld_stream(a.la[1] + slot);
                        lz = ld_stream(a.la[2] + slot);
                    }
                    Affine P;
                    if (in_prev) {
                        P.r0 = s_g[prv][0][p - prevA];
                        P.r1 = s_g[prv][1][p - prevA];
                        P.r2 = s_g[prv][2][p - prevA];
                    } else if (p != FYX_NONE) {
                        P.r0 = a.G[0][p];
                        P.r1 = a.G[1][p];
                        P.r2 = a.G[2][p];
                    } else {
                        P = affine_identity();
                    }
                    Gm = affine_mul(P, L);
                    st_stream(a.G[0] + slot, Gm.r0);
                    st_stream(a.G[1] + slot, Gm.r1);
                    st_stream(a.G[2] + slot, Gm.r2);
                    wx = aabb_transform_row(Gm.r0, lx, ly, lz);
                    wy = aabb_transform_row(Gm.r1, lx, ly, lz);
                    wz = aabb_transform_row(Gm.r2, lx, ly, lz);
                    st_stream(a.wa[0] + slot, wx);
                    st_stream(a.wa[1] + slot, wy);
                    st_stream(a.wa[2] + slot, wz);
                } else {
                    // clean node: its children may be dirty and need its (unchanged) matrix
                    Gm.r0 = a.G[0][slot];
                    Gm.r1 = a.G[1][slot];
                    Gm.r2 = a.G[2][slot];
                    if (NFT >= 0) {
                        wx = ld_stream(a.wa[0] + slot);
                        wy = ld_stream(a.wa[1] + slot);
                        wz = ld_stream(a.wa[2] + slot);
                    }
                }
                s_g[cur][0][me] = Gm.r0;
                s_g[cur][1][me] = Gm.r1;
                s_g[cur][2][me] = Gm.r2;
            }
            if (NFT >= 0) {
                const bool cand = valid && !(nf & F_SKINNED);
                const uint32_t mask = cand ? a.mask[slot] : 0u;
                const uint32_t vis_bits = cull_warp<(NFT > 0 ? NFT : 0), false>(cand, nf, mask, wx, wy, wz, cp, nullptr);
                if (DEFER) {
                    if (valid) a.vis[slot] = (uint8_t)vis_bits;
                } else {
                    const uint32_t gi = vis_bits ? a.gidx[slot] : 0u;
                    compact_emit<(NFT > 0 ? NFT : 0)>(vis_bits, gi, slot, cp);
                }
            }
        }
        __syncthreads(); // this level's rows are complete (and the previous level's are no longer read)
        prevA = r.x;
        prevB = r.y;
    }
}

// ------------------------------------------------------------------------------------------------
// Deferred compaction.  With the cull fused into the level kernels, the compaction (ballots, shared-memory prefix, one
// atomic per CTA and frustum, three CTA-wide barriers) sat at the end of a 900-instruction thread and every warp of a CTA
// waited for the slowest one.  Here the level kernels store ONE byte per node (its visible bits) and this small pass —
// 1 B read per node, gidx only where something is visible — turns the byte column into the lists: a thread takes 8
// consecutive slots, a warp 256, one atomicAdd per (warp, frustum with anything visible).  Skinned meshes are emitted by
// k_fold_bones (their byte is 0).  Order inside a list stays unspecified.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) k_compact_vis(const NodeArrays a, const CullParams cp)
{
    pdl_trigger();
    pdl_wait();
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t first = ((uint64_t)blockIdx.x * kBlock + threadIdx.x) * 8u;
    unsigned long long v = 0ull;
    if (first + 8u <= a.cap) {
        v = *reinterpret_cast<const unsigned long long *>(a.vis + first); // the column is 256-byte aligned: 8-byte loads are
    } else if (first < a.cap) {
        for (uint32_t j = 0; j < 8u && first + j < a.cap; ++j) v |= (unsigned long long)a.vis[first + j] << (8u * j);
    }
    uint32_t frusta = 0u; // frusta this thread has entries for
    {
        unsigned long long t = v;
        t |= t >> 32;
        t |= t >> 16;
        t |= t >> 8;
        frusta = (uint32_t)(t & 0xFFu);
    }
    uint32_t m = __reduce_or_sync(0xFFFFFFFFu, frusta);
    if (!m) return;
    uint32_t gi[8];
    if (v) {
#pragma unroll
        for (int j = 0; j < 8; ++j) gi[j] = (first + j < a.cap) ? a.gidx[first + j] : 0u;
    }
    while (m) {
        const int f = __ffs(m) - 1;
        m &= m - 1u;
        const unsigned long long sel = (v >> f) & 0x0101010101010101ull; // byte j = node j visible in f
        const uint32_t cnt = (uint32_t)__popcll(sel);
        uint32_t incl = cnt; // inclusive warp scan
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= (uint32_t)d) incl += t;
        }
        const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
        uint32_t base = 0u;
        if (lane == 0) base = atomicAdd(cp.counts + f * kCountStride, total);
        base = __shfl_sync(0xFFFFFFFFu, base, 0) + incl - cnt;
        if (cnt) {
            uint32_t k = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if ((sel >> (8 * j)) & 1ull) {
                    cp.out[f][base + k] = gi[j];
                    if (cp.out_slot[f]) cp.out_slot[f][base + k] = (uint32_t)(first + j);
                    ++k;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Stand-alone cull over all slots (static scene / extra passes: every shadow pass re-runs the cull
// with its own frustum, renderer/shadow/*.rs).  32 B read per node + 4 B per visible entry.
// ------------------------------------------------------------------------------------------------
// prune != nullptr: one launch per hierarchy level [lo, hi) — a node is hidden for the frusta in which an ancestor pruned the
// DFS: a statically batched mesh that is rendered (RdcControlFlow::Break, scene/mesh/mod.rs:725; renderer/bundle.rs:996-1001)
// or, through lodp, a LOD object out of range.  prune[slot] = frusta hidden for the node's children.
template <int NFT, int VAR>
__global__ void __launch_bounds__(kBlock) k_cull(const NodeArrays a, const CullParams cp, const uint32_t *lodp, const uint32_t lo, const uint32_t hi,
                                                 uint32_t *prune)
{
    constexpr bool PRE = (VAR & 1) != 0;
    __shared__ __align__(16) unsigned char s_pref[PRE ? sizeof(PrefTable) : 16];
    PrefTable *T = reinterpret_cast<PrefTable *>(s_pref);
    if (PRE) {
        pref_fill(*T, cp, NFT > 0 ? NFT : cp.nf);
        __syncthreads();
    }
    const uint32_t slot = lo + blockIdx.x * kBlock + threadIdx.x;
    const bool valid = slot < hi;
    uint32_t nf = 0u, mask = 0u;
    float2 wx = make_float2(0.f, 0.f), wy = wx, wz = wx;
    if (valid) {
        nf = a.flags[slot];
        mask = a.mask[slot];
        wx = ld_stream(a.wa[0] + slot);
        wy = ld_stream(a.wa[1] + slot);
        wz = ld_stream(a.wa[2] + slot);
    }
    uint32_t vis_bits = (VAR & 32) ? cull_warp_conv<NFT>(valid, nf, mask, wx, wy, wz, cp) : cull_warp<NFT, PRE>(valid, nf, mask, wx, wy, wz, cp, T);
    uint32_t hidden = 0u;
    if (valid && (lodp || prune)) {
        if (lodp) hidden = lodp[slot]; // frusta whose LOD filter hides the node or one of its ancestors
        if (prune) {
            const uint32_t p = a.parent[slot];
            if (p != FYX_NONE) hidden |= prune[p];
        }
        vis_bits &= ~hidden;
        if (prune) prune[slot] = hidden | ((nf & FYX_NODE_STATIC_BATCH) ? vis_bits : 0u);
    }
    const uint32_t gi = vis_bits ? a.gidx[slot] : 0u;
    if (VAR & 2) compact_emit_warp(vis_bits, gi, slot, cp);
    else compact_emit<NFT>(vis_bits, gi, slot, cp);
}

// ------------------------------------------------------------------------------------------------
// Light list (N4): the collect_lights loop of RenderDataBundleStorage::from_graph (renderer/bundle.rs:926-974) — for every
// frustum the light nodes whose world box it intersects and that are globally visible and enabled.  Lights are few:
// one pass over the flag column (4 B/node), one atomic per visible (light, frustum).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) k_cull_lights(const NodeArrays a, const CullParams cp, uint32_t *const *out, uint32_t *counts)
{
    const uint32_t slot = blockIdx.x * kBlock + threadIdx.x;
    if (slot >= a.cap) return;
    const uint32_t nf = a.flags[slot];
    constexpr uint32_t need = FYX_NODE_ALIVE | FYX_NODE_LIGHT | FYX_NODE_GLOBAL_VISIBILITY | FYX_NODE_GLOBAL_ENABLED;
    if ((nf & need) != need) return;
    const float2 wx = a.wa[0][slot], wy = a.wa[1][slot], wz = a.wa[2][slot];
    PackedConsts kc;
    kc.one = make_float2(cp.one, cp.one);
    kc.negzero = make_float2(cp.negzero, cp.negzero);
    const bool tame = aabb_is_tame(wx, wy, wz);
    const uint32_t gi = a.gidx[slot];
    for (int f = 0; f < cp.nf; ++f)
        if (frustum_intersects_aabb(cp.f[f], wx, wy, wz, kc, tame)) out[f][atomicAdd(counts + f * kCountStride, 1u)] = gi;
}

// ------------------------------------------------------------------------------------------------
// Skinned-mesh world AABB: the "special case for skinned meshes" of Mesh::on_global_transform_changed
// (scene/mesh/mod.rs:673-684): world_aabb.add_point(bone.global_position()) for every bone of every
// surface, strict </> updates in bone order (aabb.rs:86-106).  Runs after all levels (bones may be deeper than the mesh node);
// only meshes in a changed sub-tree are refreshed, as in the reference.  With (NFT >= 0) the skinned
// nodes are also culled here (they were skipped by the level kernels).
// ------------------------------------------------------------------------------------------------
// One WARP per skinned mesh: lanes take the bones round-robin, then the per-lane candidates are merged with
// a shuffle reduction keyed (value, position in the bone list) so that among numerically equal bounds
// (only -0 / +0 can differ in bits) the first one in the reference's order wins — the result is the
// reference's sequential add_point loop, bit for bit.
__device__ __forceinline__ void fold_min(float &v, uint32_t &k, const float ov, const uint32_t ok)
{
    if (ov < v || (ov == v && ok < k)) { v = ov; k = ok; }
}
__device__ __forceinline__ void fold_max(float &v, uint32_t &k, const float ov, const uint32_t ok)
{
    if (ov > v || (ov == v && ok < k)) { v = ov; k = ok; }
}

// one warp = one skinned mesh (i): refreshes the world box (all lanes return it) and reads what the cull needs
// Every table load that does not depend on another one is issued up front (mesh slot, bone range, the first two rounds of
// bone slots): three dependent memory round trips per mesh (index -> bone slot -> bone matrix) instead of five.
__device__ __forceinline__ void fold_mesh(const NodeArrays &a, const FoldArrays &fa, const uint32_t i, const uint32_t lane, uint32_t &nf_out,
                                          float2 &wx, float2 &wy, float2 &wz)
{
    const uint32_t slot = fa.node_slot[i];
    const uint32_t b0 = fa.bone_begin[i], b1 = fa.bone_begin[i + 1];
    uint32_t bs_pre[2], si_pre[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const uint32_t b = b0 + lane + 32u * r;
        bs_pre[r] = (b < b1) ? fa.bone_slot[b] : FYX_NONE;
        si_pre[r] = (b < b1 && fa.stale_idx) ? fa.stale_idx[b] : FYX_NONE;
    }
    const uint32_t nf = a.flags[slot];
    nf_out = nf;
    wx = a.wa[0][slot];
    wy = a.wa[1][slot];
    wz = a.wa[2][slot];
    if (!(nf & F_DIRTY)) return;
    // candidates start as the transformed box (order key 0 = "already there"); bones get keys 1..
    float mnx = wx.x, mny = wy.x, mnz = wz.x, mxx = wx.y, mxy = wy.y, mxz = wz.y;
    uint32_t kmnx = 0, kmny = 0, kmnz = 0, kmxx = 0, kmxy = 0, kmxz = 0;
    auto add_bone = [&](const uint32_t b, const uint32_t bs, const uint32_t si) {
        if (bs == FYX_NONE) return; // try_borrow failed ⇒ skipped
        float px, py, pz; // global_position()
        if (si != FYX_NONE) { // visited after the mesh by the reference's DFS: its value from before this update
            const float4 o = fa.stale_pos[si];
            px = o.x; py = o.y; pz = o.z;
        } else {
            px = a.G[0][bs].w;
            py = a.G[1][bs].w;
            pz = a.G[2][bs].w;
        }
        const uint32_t key = b - b0 + 1u;
        // within a lane keys increase, so the strict compares keep the earliest of equal values
        if (px < mnx) { mnx = px; kmnx = key; }
        if (py < mny) { mny = py; kmny = key; }
        if (pz < mnz) { mnz = pz; kmnz = key; }
        if (px > mxx) { mxx = px; kmxx = key; }
        if (py > mxy) { mxy = py; kmxy = key; }
        if (pz > mxz) { mxz = pz; kmxz = key; }
    };
#pragma unroll
    for (int r = 0; r < 2; ++r) add_bone(b0 + lane + 32u * r, bs_pre[r], si_pre[r]);
    for (uint32_t b = b0 + lane + 64u; b < b1; b += 32)
        add_bone(b, fa.bone_slot[b], fa.stale_idx ? fa.stale_idx[b] : FYX_NONE);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        fold_min(mnx, kmnx, __shfl_xor_sync(0xFFFFFFFFu, mnx, o), __shfl_xor_sync(0xFFFFFFFFu, kmnx, o));
        fold_min(mny, kmny, __shfl_xor_sync(0xFFFFFFFFu, mny, o), __shfl_xor_sync(0xFFFFFFFFu, kmny, o));
        fold_min(mnz, kmnz, __shfl_xor_sync(0xFFFFFFFFu, mnz, o), __shfl_xor_sync(0xFFFFFFFFu, kmnz, o));
        fold_max(mxx, kmxx, __shfl_xor_sync(0xFFFFFFFFu, mxx, o), __shfl_xor_sync(0xFFFFFFFFu, kmxx, o));
        fold_max(mxy, kmxy, __shfl_xor_sync(0xFFFFFFFFu, mxy, o), __shfl_xor_sync(0xFFFFFFFFu, kmxy, o));
        fold_max(mxz, kmxz, __shfl_xor_sync(0xFFFFFFFFu, mxz, o), __shfl_xor_sync(0xFFFFFFFFu, kmxz, o));
    }
    wx = make_float2(mnx, mxx);
    wy = make_float2(mny, mxy);
    wz = make_float2(mnz, mxz);
    if (lane == 0) {
        a.wa[0][slot] = wx;
        a.wa[1][slot] = wy;
        a.wa[2][slot] = wz;
    }
}

// One warp per skinned mesh folds the bones; the cull of the CTA's kBlock/32 meshes is then run by the first lanes of warp 0,
// one mesh per LANE (the multi-frustum predicate is a long dependent chain: run by lane 0 of every warp it cost eight times the
// issue slots), and warp 0 emits the entries.
template <int NFT>
__global__ void __launch_bounds__(kBlock) k_fold_bones(const NodeArrays a, const FoldArrays fa, const CullParams cp)
{
    pdl_trigger();
    pdl_wait();
    constexpr int kWarps = kBlock / 32;
    __shared__ float2 s_box[3][kWarps];
    __shared__ uint32_t s_nf[kWarps];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t i = blockIdx.x * kWarps + warp; // mesh = warp
    uint32_t nf = 0u;
    float2 wx = make_float2(0.f, 0.f), wy = wx, wz = wx;
    if (i < fa.n) fold_mesh(a, fa, i, lane, nf, wx, wy, wz);
    if (NFT < 0) return;
    if (lane == 0) {
        s_box[0][warp] = wx;
        s_box[1][warp] = wy;
        s_box[2][warp] = wz;
        s_nf[warp] = (i < fa.n) ? nf : 0u;
    }
    __syncthreads();
    if (warp != 0) return;
    uint32_t vis_bits = 0u, gi = 0u, slot = 0u;
    const uint32_t m = blockIdx.x * kWarps + lane; // lane l of warp 0 culls the mesh of warp l
    if (lane < kWarps && m < fa.n) {
        PackedConsts kc;
        kc.one = make_float2(cp.one, cp.one);
        kc.negzero = make_float2(cp.negzero, cp.negzero);
        slot = fa.node_slot[m];
        const float2 bx = s_box[0][lane], by = s_box[1][lane], bz = s_box[2][lane];
        vis_bits = cull_bits<(NFT > 0 ? NFT : 0)>(s_nf[lane], a.mask[slot], bx, by, bz, cp, kc, aabb_is_tame(bx, by, bz), 0xFFFFFFFFu);
        if (vis_bits) gi = a.gidx[slot];
    }
    compact_emit_warp(vis_bits, gi, slot, cp);
}

// positions of the "late" bones (see FoldArrays) as stored before the update starts
__global__ void __launch_bounds__(kBlock) k_snapshot_bones(const NodeArrays a, const uint32_t n_late, const uint32_t *late_slot,
                                                           float4 *stale_pos)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= n_late) return;
    const uint32_t s = late_slot[e];
    stale_pos[e] = make_float4(a.G[0][s].w, a.G[1][s].w, a.G[2][s].w, 0.0f);
}

// ------------------------------------------------------------------------------------------------
// Bone palette: SurfaceInstanceData::bone_matrices (scene/mesh/mod.rs:781-793):
// P[k] = bone_k.global_transform() * bone_k.inv_bind_pose_transform(), identity for an invalid
// handle.  One thread per (surface, bone) entry; G is gathered by bone slot, inv_bind streams.
// Output: column-major mat4 (the layout write_uniforms copies into the UBO, renderer/bundle.rs:484-496).
// Algorithmic bytes per bone: 196 (G 64 + inv_bind 64 + idx 4 + P 64); moved: 48 + 48 + 4 + 64.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void palette_entry(const NodeArrays &a, const SkinArrays &sk, const uint32_t e)
{
    const uint32_t bs = sk.bone_slot[e];
    Affine P;
    if (bs != FYX_NONE) {
        Affine Gm, IB;
        Gm.r0 = a.G[0][bs];
        Gm.r1 = a.G[1][bs];
        Gm.r2 = a.G[2][bs];
        IB.r0 = ld_stream(sk.ib[0] + e);
        IB.r1 = ld_stream(sk.ib[1] + e);
        IB.r2 = ld_stream(sk.ib[2] + e);
        P = affine_mul(Gm, IB);
    } else {
        P = affine_identity();
    }
    float4 *o = reinterpret_cast<float4 *>(sk.palette + 16 * (size_t)e);
    o[0] = make_float4(P.r0.x, P.r1.x, P.r2.x, 0.0f);
    o[1] = make_float4(P.r0.y, P.r1.y, P.r2.y, 0.0f);
    o[2] = make_float4(P.r0.z, P.r1.z, P.r2.z, 0.0f);
    o[3] = make_float4(P.r0.w, P.r1.w, P.r2.w, 1.0f);
}

__global__ void __launch_bounds__(kBlock) k_palette(const NodeArrays a, const SkinArrays sk)
{
    pdl_trigger();
    pdl_wait();
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e < sk.n_entries) palette_entry(a, sk, e);
}

// ------------------------------------------------------------------------------------------------
// Linear-blend skinning.  Positions: the skinned branch of Mesh::accurate_world_bounding_box
// (scene/mesh/mod.rs:501-522): acc = 0; for k in 0..4: acc += P[idx_k].transform_point(p) * w_k, where
// transform_point = ((m_i0*x + m_i1*y) + m_i2*z) + m_i3, then / n with n = row3·p + m33 — exactly 1
// for the affine palette and finite p, so the division is the identity and is skipped.  Normals:
// standard.shader:192-195, acc += (mat3(P[idx_k]) * n) * w_k in the same order.
//
// * Each thread owns 4 consecutive vertices.  Inputs live in blocks of 128 vertices x 11 rows of 512 B
//   (x, y, z, nx, ny, nz, w0..w3, indices; fyx_internal.h): a warp reads a row with ONE coalesced 512 B
//   access and each 32 B sector exactly once (the packed-xyz layout made every sector travel L2->SM
//   twice).  Outputs are packed xyz streams, 3 + 3 128-bit stores per thread.
// * Arithmetic uses Blackwell's packed FP32 pipe (mul.rn.f32x2 / add.rn.f32x2 via __fmul2_rn /
//   __fadd2_rn: two independently rounded f32 results per issue slot).  The kernel is issue-bound
//   (ncu: 8.6 warp-instructions per vertex), and FMA contraction is forbidden, so halving the FP
//   instruction count is the lever.  Pairs: (x,y) of the position, (x,y) of the normal, and
//   (position.z, normal.z) — same op order per element as the scalar reference.
// * The surface's palette sits in shared memory as three float4 planes laid out for those pairs:
//     A = (m00,m10,m01,m11)  B = (m02,m12,m03,m13)  Z = (m20,m21,m22,m23)
//   (the z pair multiplies the register pair (p,n) by a scalar-broadcast operand of FFMA2, so the third
//   row needs no duplication), each plane REPLICATED C times: bone b of copy c at float4 index plane*PL + c*S + b with S = 1 mod 8,
//   PL = C*S.  A 128-bit shared load is served per quarter-warp; lane l reads copy (l - b) mod C,
//   which puts it in bank group (plane*PL + l) mod 8: conflict-free for C = 8 whatever the bone
//   indices are (with one copy, 57 % of the shared-memory wavefronts were conflict replays).
// Algorithmic bytes per vertex: 44 read + 24 written = 68.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 lo2(const float4 v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi2(const float4 v) { return make_float2(v.z, v.w); }

// palette (column-major mat4 in global memory) → the four replicated planes
template <int S, int LOG2C>
__device__ __forceinline__ void skin_fill_palette(float4 *s_pal, const float *palette, const uint32_t bone_off, const uint32_t n_bones)
{
    constexpr int C = 1 << LOG2C;
    constexpr int PL = S * C;
    for (uint32_t b = threadIdx.x; b < n_bones; b += kBlock) {
        const float4 *m = reinterpret_cast<const float4 *>(palette + 16 * (size_t)(bone_off + b));
        const float4 c0 = m[0], c1 = m[1], c2 = m[2], c3 = m[3];
        const float4 A = make_float4(c0.x, c0.y, c1.x, c1.y);
        const float4 B = make_float4(c2.x, c2.y, c3.x, c3.y);
        const float4 Z = make_float4(c0.z, c1.z, c2.z, c3.z);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            s_pal[0 * PL + c * S + b] = A;
            s_pal[1 * PL + c * S + b] = B;
            s_pal[2 * PL + c * S + b] = Z;
        }
    }
}

// four vertices (one thread's group) from registers to the two output streams; TAN: also their tangents to the third
// (standard.shader:197-200 skins inputTangent.xyz as the normal, acc += (mat3(P[idx_k]) * t) * w_k, k in order).  The
// tangent reuses the palette rows the position and normal just read: (tx, ty) go through the packed pipe as the normal's
// (x, y), tz is the scalar third row, r_z = (m_20*tx + m_21*ty) + m_22*tz (one rounding per product and sum).
template <int S, int LOG2C, bool TAN = false>
__device__ __forceinline__ void skin_quad(const float4 *s_pal, const uint32_t lane, const float4 x4, const float4 y4, const float4 z4,
                                          const float4 nx4, const float4 ny4, const float4 nz4, const float4 w0, const float4 w1,
                                          const float4 w2, const float4 w3, const uint4 iq, float4 *po, float4 *no,
                                          const PackedConsts kc, const float4 tx4 = float4{}, const float4 ty4 = float4{},
                                          const float4 tz4 = float4{}, float4 *to = nullptr)
{
    constexpr int C = 1 << LOG2C;
    constexpr int PL = S * C;
    const float px[4] = {x4.x, x4.y, x4.z, x4.w}, py[4] = {y4.x, y4.y, y4.z, y4.w}, pz[4] = {z4.x, z4.y, z4.z, z4.w};
    const float nx[4] = {nx4.x, nx4.y, nx4.z, nx4.w}, ny[4] = {ny4.x, ny4.y, ny4.z, ny4.w}, nz[4] = {nz4.x, nz4.y, nz4.z, nz4.w};
    const float tx[4] = {tx4.x, tx4.y, tx4.z, tx4.w}, ty[4] = {ty4.x, ty4.y, ty4.z, ty4.w}, tz[4] = {tz4.x, tz4.y, tz4.z, tz4.w};
    // w_k holds weight k of the four vertices
    const float wk4[4][4] = {{w0.x, w1.x, w2.x, w3.x}, {w0.y, w1.y, w2.y, w3.y}, {w0.z, w1.z, w2.z, w3.z}, {w0.w, w1.w, w2.w, w3.w}};
    const uint32_t iv[4] = {iq.x, iq.y, iq.z, iq.w};
    float ox[4], oy[4], oz[4], mx[4], my[4], mz[4], ux[4], uy[4], uz[4];
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        const float2 pxx = make_float2(px[v], px[v]), pyy = make_float2(py[v], py[v]), pzz = make_float2(pz[v], pz[v]);
        const float2 nxx = make_float2(nx[v], nx[v]), nyy = make_float2(ny[v], ny[v]), nzz = make_float2(nz[v], nz[v]);
        const float2 pnx = make_float2(px[v], nx[v]), pny = make_float2(py[v], ny[v]), pnz = make_float2(pz[v], nz[v]);
        float2 acc_p = make_float2(0.0f, 0.0f), acc_n = make_float2(0.0f, 0.0f), acc_z = make_float2(0.0f, 0.0f);
        float2 acc_t = make_float2(0.0f, 0.0f);
        float acc_tz = 0.0f;
        const float *wk = wk4[v];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t bone = (iv[v] >> (8 * k)) & 0xFFu;
            const float4 *row = s_pal + (((lane - bone) & (uint32_t)(C - 1)) * S + bone);
            const float4 A = row[0], B = row[PL], Z = row[2 * PL];
            const float2 ww = make_float2(wk[k], wk[k]);
            // (tx, ty) = ((m_i0*x + m_i1*y) + m_i2*z) + m_i3, i = 0,1
            const float2 t = add2(add2(add2(mul2(lo2(A), pxx, kc), mul2(hi2(A), pyy, kc), kc), mul2(lo2(B), pzz, kc), kc), hi2(B), kc);
            acc_p = add2(acc_p, mul2(t, ww, kc), kc);
            // (rx, ry) = (m_i0*nx + m_i1*ny) + m_i2*nz
            const float2 r = add2(add2(mul2(lo2(A), nxx, kc), mul2(hi2(A), nyy, kc), kc), mul2(lo2(B), nzz, kc), kc);
            acc_n = add2(acc_n, mul2(r, ww, kc), kc);
            // (tz', rz) = (m_20*{x,nx} + m_21*{y,ny}) + m_22*{z,nz};  tz = tz' + m_23
            float2 z = add2(add2(mul2(pnx, make_float2(Z.x, Z.x), kc), mul2(pny, make_float2(Z.y, Z.y), kc), kc), mul2(pnz, make_float2(Z.z, Z.z), kc), kc);
            z.x = FYX_ADD(z.x, Z.w);
            acc_z = add2(acc_z, mul2(z, ww, kc), kc);
            if (TAN) {
                // tangent (sx, sy) = (m_i0*tx + m_i1*ty) + m_i2*tz;  sz = (m_20*tx + m_21*ty) + m_22*tz
                const float2 txx = make_float2(tx[v], tx[v]), tyy = make_float2(ty[v], ty[v]), tzz = make_float2(tz[v], tz[v]);
                const float2 sxy = add2(add2(mul2(lo2(A), txx, kc), mul2(hi2(A), tyy, kc), kc), mul2(lo2(B), tzz, kc), kc);
                acc_t = add2(acc_t, mul2(sxy, ww, kc), kc);
                const float sz = FYX_ADD(FYX_ADD(FYX_MUL(Z.x, tx[v]), FYX_MUL(Z.y, ty[v])), FYX_MUL(Z.z, tz[v]));
                acc_tz = FYX_ADD(acc_tz, FYX_MUL(sz, wk[k]));
            }
        }
        ox[v] = acc_p.x; oy[v] = acc_p.y; oz[v] = acc_z.x;
        mx[v] = acc_n.x; my[v] = acc_n.y; mz[v] = acc_z.y;
        ux[v] = acc_t.x; uy[v] = acc_t.y; uz[v] = acc_tz;
    }
    st_stream(po + 0, make_float4(ox[0], oy[0], oz[0], ox[1]));
    st_stream(po + 1, make_float4(oy[1], oz[1], ox[2], oy[2]));
    st_stream(po + 2, make_float4(oz[2], ox[3], oy[3], oz[3]));
    st_stream(no + 0, make_float4(mx[0], my[0], mz[0], mx[1]));
    st_stream(no + 1, make_float4(my[1], mz[1], mx[2], my[2]));
    st_stream(no + 2, make_float4(mz[2], mx[3], my[3], mz[3]));
    if (TAN) {
        st_stream(to + 0, make_float4(ux[0], uy[0], uz[0], ux[1]));
        st_stream(to + 1, make_float4(uy[1], uz[1], ux[2], uy[2]));
        st_stream(to + 2, make_float4(uz[2], ux[3], uy[3], uz[3]));
    }
}

// two vertices (half of a four-vertex group) per thread: 22 input registers instead of 44 — k_skin2 trades wider loads for
// more resident warps (k_skin sits at 24 warps per SM with 80 registers and is bound by load latency, not by bandwidth)
template <int S, int LOG2C>
__device__ __forceinline__ void skin_pair(const float4 *s_pal, const uint32_t lane, const float2 x2, const float2 y2, const float2 z2, const float2 nx2,
                                          const float2 ny2, const float2 nz2, const float2 w0, const float2 w1, const float2 w2, const float2 w3,
                                          const uint2 iq, float2 *po, float2 *no, const PackedConsts kc)
{
    constexpr int C = 1 << LOG2C;
    constexpr int PL = S * C;
    const float px[2] = {x2.x, x2.y}, py[2] = {y2.x, y2.y}, pz[2] = {z2.x, z2.y};
    const float nx[2] = {nx2.x, nx2.y}, ny[2] = {ny2.x, ny2.y}, nz[2] = {nz2.x, nz2.y};
    const float wk2[2][4] = {{w0.x, w1.x, w2.x, w3.x}, {w0.y, w1.y, w2.y, w3.y}};
    const uint32_t iv[2] = {iq.x, iq.y};
    float ox[2], oy[2], oz[2], mx[2], my[2], mz[2];
#pragma unroll
    for (int v = 0; v < 2; ++v) {
        const float2 pxx = make_float2(px[v], px[v]), pyy = make_float2(py[v], py[v]), pzz = make_float2(pz[v], pz[v]);
        const float2 nxx = make_float2(nx[v], nx[v]), nyy = make_float2(ny[v], ny[v]), nzz = make_float2(nz[v], nz[v]);
        const float2 pnx = make_float2(px[v], nx[v]), pny = make_float2(py[v], ny[v]), pnz = make_float2(pz[v], nz[v]);
        float2 acc_p = make_float2(0.0f, 0.0f), acc_n = make_float2(0.0f, 0.0f), acc_z = make_float2(0.0f, 0.0f);
        const float *wk = wk2[v];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t bone = (iv[v] >> (8 * k)) & 0xFFu;
            const float4 *row = s_pal + (((lane - bone) & (uint32_t)(C - 1)) * S + bone);
            const float4 A = row[0], B = row[PL], Z = row[2 * PL];
            const float2 ww = make_float2(wk[k], wk[k]);
            const float2 t = add2(add2(add2(mul2(lo2(A), pxx, kc), mul2(hi2(A), pyy, kc), kc), mul2(lo2(B), pzz, kc), kc), hi2(B), kc);
            acc_p = add2(acc_p, mul2(t, ww, kc), kc);
            const float2 r = add2(add2(mul2(lo2(A), nxx, kc), mul2(hi2(A), nyy, kc), kc), mul2(lo2(B), nzz, kc), kc);
            acc_n = add2(acc_n, mul2(r, ww, kc), kc);
            float2 z = add2(add2(mul2(pnx, make_float2(Z.x, Z.x), kc), mul2(pny, make_float2(Z.y, Z.y), kc), kc), mul2(pnz, make_float2(Z.z, Z.z), kc), kc);
            z.x = FYX_ADD(z.x, Z.w);
            acc_z = add2(acc_z, mul2(z, ww, kc), kc);
        }
        ox[v] = acc_p.x; oy[v] = acc_p.y; oz[v] = acc_z.x;
        mx[v] = acc_n.x; my[v] = acc_n.y; mz[v] = acc_z.y;
    }
    st_stream(po + 0, make_float2(ox[0], oy[0]));
    st_stream(po + 1, make_float2(oz[0], ox[1]));
    st_stream(po + 2, make_float2(oy[1], oz[1]));
    st_stream(no + 0, make_float2(mx[0], my[0]));
    st_stream(no + 1, make_float2(mz[0], mx[1]));
    st_stream(no + 2, make_float2(my[1], mz[1]));
}

template <int S, int LOG2C, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) k_skin2(const SkinArrays sk, const SkinTile *__restrict__ tiles, const uint32_t n_tiles, const float one,
                                                      const float negzero)
{
    extern __shared__ float4 smem[];
    float4 *const s_pal = smem;
    PackedConsts kc;
    kc.one = make_float2(one, one);
    kc.negzero = make_float2(negzero, negzero);
    const SkinTile T = tiles[blockIdx.x];
    pdl_wait(); // the palettes come from k_palette
    skin_fill_palette<S, LOG2C>(s_pal, sk.palette, T.bone_off, T.n_bones);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t h = threadIdx.x; h < 2u * T.n_quads; h += kBlock) {
        const size_t quad = (size_t)T.quad_start + (h >> 1);
        const float2 *row = reinterpret_cast<const float2 *>(sk.vblk + (quad >> 5) * kVblkStride + (quad & 31)) + (h & 1u);
        const float2 x2 = ld_stream(row + 0 * 64), y2 = ld_stream(row + 1 * 64), z2 = ld_stream(row + 2 * 64);
        const float2 nx2 = ld_stream(row + 3 * 64), ny2 = ld_stream(row + 4 * 64), nz2 = ld_stream(row + 5 * 64);
        const float2 w0 = ld_stream(row + 6 * 64), w1 = ld_stream(row + 7 * 64), w2 = ld_stream(row + 8 * 64), w3 = ld_stream(row + 9 * 64);
        const float2 iqf = ld_stream(row + 10 * 64);
        const uint2 iq = make_uint2(__float_as_uint(iqf.x), __float_as_uint(iqf.y));
        const size_t pair = 2 * quad + (h & 1u); // index of the vertex pair: 6 floats = 3 float2 per stream
        skin_pair<S, LOG2C>(s_pal, lane, x2, y2, z2, nx2, ny2, nz2, w0, w1, w2, w3, iq, reinterpret_cast<float2 *>(sk.opos) + 3 * pair,
                            reinterpret_cast<float2 *>(sk.onrm) + 3 * pair, kc);
    }
}

// N4: blend shapes ahead of the skinning (standard.shader:167-173): for i in 0..blendShapesCount:
//   inputPosition.xyz += offsets.position * weight;  inputNormal += offsets.normal * weight
// in shape order, offsets = the f16 texels of BlendShapesContainer::from_lists (scene/mesh/surface.rs:92-218, exact in
// f32), weight = BlendShape::weight / 100 (scene/mesh/mod.rs:794-798); one rounding per product and per sum.
// 12 more bytes read per vertex and shape.  The four vertices of a thread come as 4 halfs per row.
__device__ __forceinline__ void bs_axpy(float4 &v, const uint2 h, const float w)
{
    const __half2 a = *reinterpret_cast<const __half2 *>(&h.x), b = *reinterpret_cast<const __half2 *>(&h.y);
    const float2 fa = __half22float2(a), fb = __half22float2(b);
    v.x = FYX_ADD(v.x, FYX_MUL(fa.x, w));
    v.y = FYX_ADD(v.y, FYX_MUL(fa.y, w));
    v.z = FYX_ADD(v.z, FYX_MUL(fb.x, w));
    v.w = FYX_ADD(v.w, FYX_MUL(fb.y, w));
}

__device__ __forceinline__ void apply_blend_shapes(const SkinArrays &sk, const SkinTile &T, const uint32_t q, float4 &x4, float4 &y4, float4 &z4,
                                                   float4 &nx4, float4 &ny4, float4 &nz4)
{
    const uint32_t e = T.local_quad0 + q;
    const uint2 *r0 = sk.bs + ((size_t)T.bs_off + (e >> 5)) * kBsBlockU2 + (e & 31u);
    const size_t shape_stride = (size_t)T.bs_blocks * kBsBlockU2;
    for (uint32_t sidx = 0; sidx < T.n_shapes; ++sidx) {
        const float w = sk.bs_w[T.w_off + sidx];
        const uint2 *r = r0 + sidx * shape_stride;
        const uint2 hx = r[0 * 32], hy = r[1 * 32], hz = r[2 * 32], hnx = r[3 * 32], hny = r[4 * 32], hnz = r[5 * 32];
        bs_axpy(x4, hx, w);
        bs_axpy(y4, hy, w);
        bs_axpy(z4, hz, w);
        bs_axpy(nx4, hnx, w);
        bs_axpy(ny4, hny, w);
        bs_axpy(nz4, hnz, w);
    }
}

// the tangent offsets of a tangent surface (fyx_set_skinned_tangents): halfs 6-8 of each record, added in shape order
// exactly as the normal offsets above (standard.shader:167-173 adds offsets.tangent * weight to inputTangent.xyz)
__device__ __forceinline__ void apply_blend_shapes_tan(const SkinArrays &sk, const SkinTile &T, const uint32_t e, float4 &tx4, float4 &ty4, float4 &tz4)
{
    const uint2 *r0 = sk.bst + ((size_t)T.bst_off + (e >> 5)) * kBstBlockU2 + (e & 31u);
    const size_t shape_stride = (size_t)T.bs_blocks * kBstBlockU2;
    for (uint32_t sidx = 0; sidx < T.n_shapes; ++sidx) {
        const float w = sk.bs_w[T.w_off + sidx];
        const uint2 *r = r0 + sidx * shape_stride;
        const uint2 htx = r[0 * 32], hty = r[1 * 32], htz = r[2 * 32];
        bs_axpy(tx4, htx, w);
        bs_axpy(ty4, hty, w);
        bs_axpy(tz4, htz, w);
    }
}

// BlendShapesContainer's records (9 halfs per vertex and layer: position, normal, tangent) -> the blocked device layout:
// halfs [H0, H0 + NH) of every record into NH rows per (shape, block) (H0 = 0, NH = 6: bs; H0 = 6, NH = 3: bst)
template <int H0, int NH>
__global__ void __launch_bounds__(kBlock) k_bs_layout(const uint32_t n_verts, const uint32_t n_shapes, const uint32_t layer_stride,
                                                      const uint16_t *rec, uint16_t *dst, const uint32_t bs_blocks)
{
    const uint64_t t = (uint64_t)blockIdx.x * kBlock + threadIdx.x;
    const uint64_t per_shape = (uint64_t)bs_blocks * 128;
    if (t >= per_shape * n_shapes) return;
    const uint32_t sidx = (uint32_t)(t / per_shape), v = (uint32_t)(t % per_shape);
    uint16_t h[NH] = {};
    if (v < n_verts) {
        const uint16_t *r = rec + ((size_t)sidx * layer_stride + v) * 9 + H0;
        for (int k = 0; k < NH; ++k) h[k] = r[k];
    }
    // (shape, block) = NH rows x 32 groups x 4 halfs
    uint16_t *blk = dst + ((size_t)sidx * bs_blocks + (v >> 7)) * (NH * 32 * 4);
    const uint32_t g = (v >> 2) & 31u, j = v & 3u;
    for (int k = 0; k < NH; ++k) blk[(k * 32 + g) * 4 + j] = h[k];
}

template <int H0, int NH>
static void launch_bs_layout_t(cudaStream_t s, uint32_t n_verts, uint32_t n_shapes, uint32_t layer_stride, const uint16_t *d_records, uint2 *d_dst,
                               uint32_t bs_blocks)
{
    if (!n_shapes || !bs_blocks) return;
    k_bs_layout<H0, NH><<<(unsigned)(((uint64_t)bs_blocks * 128 * n_shapes + kBlock - 1) / kBlock), kBlock, 0, s>>>(
        n_verts, n_shapes, layer_stride, d_records, reinterpret_cast<uint16_t *>(d_dst), bs_blocks);
}

void launch_bs_layout(cudaStream_t s, uint32_t n_verts, uint32_t n_shapes, uint32_t layer_stride, const uint16_t *d_records, uint2 *d_dst, uint32_t bs_blocks)
{
    static_assert(kBsBlockU2 * 4 == 6 * 32 * 4, "6 rows of 32 groups x 4 halfs");
    launch_bs_layout_t<0, 6>(s, n_verts, n_shapes, layer_stride, d_records, d_dst, bs_blocks);
}

void launch_bs_tan_layout(cudaStream_t s, uint32_t n_verts, uint32_t n_shapes, uint32_t layer_stride, const uint16_t *d_records, uint2 *d_dst,
                          uint32_t bs_blocks)
{
    static_assert(kBstBlockU2 * 4 == 3 * 32 * 4, "3 rows of 32 groups x 4 halfs");
    launch_bs_layout_t<6, 3>(s, n_verts, n_shapes, layer_stride, d_records, d_dst, bs_blocks);
}

// One CTA per tile, inputs loaded straight into registers (LDG.128, L1-bypassing).  TAN: some surface of the context has
// tangents; whether this tile does is CTA-uniform, and a tile without them runs the same code as the TAN = false kernel.
template <int S, int LOG2C, int MINB, bool BS, bool TAN>
__global__ void __launch_bounds__(kBlock, MINB) k_skin(const SkinArrays sk, const SkinTile *__restrict__ tiles, const uint32_t n_tiles,
                                                     const float one, const float negzero)
{
    extern __shared__ float4 smem[];
    float4 *const s_pal = smem;
    PackedConsts kc;
    kc.one = make_float2(one, one);
    kc.negzero = make_float2(negzero, negzero);
    const SkinTile T = tiles[blockIdx.x];
    pdl_wait(); // the palettes come from k_palette
    skin_fill_palette<S, LOG2C>(s_pal, sk.palette, T.bone_off, T.n_bones);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t q = threadIdx.x; q < T.n_quads; q += kBlock) {
        const size_t quad = (size_t)T.quad_start + q;
        const float4 *row = sk.vblk + (quad >> 5) * kVblkStride + (quad & 31); // block, then this group's column
        float4 x4 = ld_stream(row + 0 * 32), y4 = ld_stream(row + 1 * 32), z4 = ld_stream(row + 2 * 32);
        float4 nx4 = ld_stream(row + 3 * 32), ny4 = ld_stream(row + 4 * 32), nz4 = ld_stream(row + 5 * 32);
        const float4 w0 = ld_stream(row + 6 * 32), w1 = ld_stream(row + 7 * 32), w2 = ld_stream(row + 8 * 32), w3 = ld_stream(row + 9 * 32);
        const uint4 iq = ld_stream(reinterpret_cast<const uint4 *>(row + 10 * 32));
        if (BS && T.n_shapes) apply_blend_shapes(sk, T, q, x4, y4, z4, nx4, ny4, nz4);
        if (TAN && T.tan_blk != FYX_NONE) {
            const uint32_t e = T.local_quad0 + q; // group within the surface
            const float4 *trow = sk.tblk + ((size_t)T.tan_blk + (e >> 5)) * kTblkStride + (e & 31u);
            float4 tx4 = ld_stream(trow + 0 * 32), ty4 = ld_stream(trow + 1 * 32), tz4 = ld_stream(trow + 2 * 32);
            if (BS && T.n_shapes) apply_blend_shapes_tan(sk, T, e, tx4, ty4, tz4);
            skin_quad<S, LOG2C, true>(s_pal, lane, x4, y4, z4, nx4, ny4, nz4, w0, w1, w2, w3, iq, reinterpret_cast<float4 *>(sk.opos) + 3 * quad,
                                      reinterpret_cast<float4 *>(sk.onrm) + 3 * quad, kc, tx4, ty4, tz4,
                                      reinterpret_cast<float4 *>(sk.otan) + 3 * ((size_t)T.tan_quad0 + e));
        } else {
            skin_quad<S, LOG2C>(s_pal, lane, x4, y4, z4, nx4, ny4, nz4, w0, w1, w2, w3, iq, reinterpret_cast<float4 *>(sk.opos) + 3 * quad,
                                reinterpret_cast<float4 *>(sk.onrm) + 3 * quad, kc);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_skin with TMA bulk staging (the experiment BASELINE.json's north_star names; numbers in profiles/README.md).
// The vertex input is already laid out for it: a block of 128 vertices is 5 632 contiguous bytes (11 rows x 512 B).
// Every WARP owns a ring of STAGES block buffers in shared memory and its own mbarriers: lane 0 issues one 1-D
// cp.async.bulk (global -> shared, completion counted in bytes on the mbarrier) per block, the warp waits on the
// barrier's phase parity, reads its 11 rows with conflict-free LDS.128 (lane l owns group l of the block), computes,
// stores, and refills the buffer with the block STAGES ahead.  The vertex blocks are static, so the first copies are
// issued BEFORE griddepcontrol.wait (they overlap k_palette's tail); the palette planes are then filled as in k_skin.
// Selected with FYX_SKIN_VARIANT=tma2 (4 palette copies, 2 stages, 2 CTAs/SM) or tma3 (8 copies, 3 stages, 1 CTA/SM).
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kVblkBytes = kVblkStride * sizeof(float4); // 5632

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(const uint32_t bar, const uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(const uint32_t bar, const uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(const uint32_t bar, const uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(const uint32_t dst, const void *src, const uint32_t bytes, const uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

template <int S, int LOG2C, int STAGES, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) k_skin_tma(const SkinArrays sk, const SkinTile *__restrict__ tiles, const uint32_t n_tiles,
                                                         const float one, const float negzero)
{
    constexpr int C = 1 << LOG2C;
    constexpr int W = kBlock / 32;
    constexpr uint32_t kPalBytes = (3u * S * C * sizeof(float4) + 127u) & ~127u;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4 *const s_pal = reinterpret_cast<float4 *>(smem_raw);
    unsigned char *const ring = smem_raw + kPalBytes;
    uint64_t *const bars = reinterpret_cast<uint64_t *>(ring + (size_t)W * STAGES * kVblkBytes);
    PackedConsts kc;
    kc.one = make_float2(one, one);
    kc.negzero = make_float2(negzero, negzero);
    const SkinTile T = tiles[blockIdx.x];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t b0 = T.quad_start >> 5, b1 = (T.quad_start + T.n_quads + 31u) >> 5; // blocks [b0, b1) hold the tile
    const uint32_t q_lo = T.quad_start, q_hi = T.quad_start + T.n_quads;
    unsigned char *const my_ring = ring + (size_t)warp * STAGES * kVblkBytes;
    const uint32_t my_bar = smem_u32(bars + warp * STAGES);
    if (lane == 0) {
#pragma unroll
        for (int st = 0; st < STAGES; ++st) mbar_init(my_bar + 8u * st, 1u);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    // prologue: the first STAGES blocks of this warp (static data: does not wait for the predecessor kernel)
    if (lane == 0) {
#pragma unroll
        for (int st = 0; st < STAGES; ++st) {
            const uint32_t b = b0 + warp + (uint32_t)st * W;
            if (b < b1) {
                mbar_expect_tx(my_bar + 8u * st, kVblkBytes);
                bulk_g2s(smem_u32(my_ring + (size_t)st * kVblkBytes), sk.vblk + (size_t)b * kVblkStride, kVblkBytes, my_bar + 8u * st);
            }
        }
    }
    pdl_wait(); // the palettes come from k_palette
    skin_fill_palette<S, LOG2C>(s_pal, sk.palette, T.bone_off, T.n_bones);
    __syncthreads();
    uint32_t j = 0;
    for (uint32_t b = b0 + warp; b < b1; b += W, ++j) {
        const uint32_t st = j % STAGES, parity = (j / STAGES) & 1u;
        mbar_wait(my_bar + 8u * st, parity);
        const float4 *row = reinterpret_cast<const float4 *>(my_ring + (size_t)st * kVblkBytes) + lane;
        const size_t quad = ((size_t)b << 5) + lane;
        if (quad >= q_lo && quad < q_hi) {
            const float4 x4 = row[0 * 32], y4 = row[1 * 32], z4 = row[2 * 32];
            const float4 nx4 = row[3 * 32], ny4 = row[4 * 32], nz4 = row[5 * 32];
            const float4 w0 = row[6 * 32], w1 = row[7 * 32], w2 = row[8 * 32], w3 = row[9 * 32];
            const uint4 iq = *reinterpret_cast<const uint4 *>(row + 10 * 32);
            skin_quad<S, LOG2C>(s_pal, lane, x4, y4, z4, nx4, ny4, nz4, w0, w1, w2, w3, iq, reinterpret_cast<float4 *>(sk.opos) + 3 * quad,
                                reinterpret_cast<float4 *>(sk.onrm) + 3 * quad, kc);
        }
        __syncwarp(); // every lane has read the buffer before it is refilled
        const uint32_t nb = b + (uint32_t)STAGES * W;
        if (lane == 0 && nb < b1) {
            mbar_expect_tx(my_bar + 8u * st, kVblkBytes);
            bulk_g2s(smem_u32(my_ring + (size_t)st * kVblkBytes), sk.vblk + (size_t)nb * kVblkStride, kVblkBytes, my_bar + 8u * st);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Host-facing scatter / gather between the caller's AoS-by-node-index arrays and the slot-ordered
// SoA planes.  Invalid indices are skipped (Pool::try_borrow semantics).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t resolve_slot(const uint32_t *d_idx, uint32_t e, const uint32_t *slot_of_node,
                                                 uint32_t n_nodes)
{
    const uint32_t node = d_idx ? d_idx[e] : e;
    if (node >= n_nodes) return FYX_NONE;
    return slot_of_node[node];
}

// bottom row must be bit-exactly (+0,+0,+0,1) — what Transform::calculate_local_transform writes
// (scene/transform.rs:479-536) — and all entries finite; returns false otherwise
__device__ __forceinline__ bool load_affine_rows(const float *m16, Affine &A)
{
    const float4 *c = reinterpret_cast<const float4 *>(m16);
    const float4 c0 = c[0], c1 = c[1], c2 = c[2], c3 = c[3];
    A.r0 = make_float4(c0.x, c1.x, c2.x, c3.x);
    A.r1 = make_float4(c0.y, c1.y, c2.y, c3.y);
    A.r2 = make_float4(c0.z, c1.z, c2.z, c3.z);
    const bool bottom = (__float_as_uint(c0.w) == 0u) & (__float_as_uint(c1.w) == 0u) & (__float_as_uint(c2.w) == 0u) &
                        (c3.w == 1.0f);
    return bottom & finite4(A.r0) & finite4(A.r1) & finite4(A.r2);
}

__global__ void __launch_bounds__(kBlock) k_scatter_locals(const NodeArrays a, const uint32_t count, const uint32_t *d_idx,
                                                           const float *d_m16, const uint32_t *slot_of_node,
                                                           const uint32_t n_nodes, uint32_t *d_err)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= count) return;
    const uint32_t slot = resolve_slot(d_idx, e, slot_of_node, n_nodes);
    if (slot == FYX_NONE) return;
    Affine A;
    if (!load_affine_rows(d_m16 + 16 * (size_t)e, A)) {
        atomicOr(d_err, E_NOT_AFFINE);
        return;
    }
    a.L[0][slot] = A.r0;
    a.L[1][slot] = A.r1;
    a.L[2][slot] = A.r2;
    atomicOr(a.flags + slot, F_DIRTY_SELF); // NodeMessageKind::TransformChanged
}

// Transform::calculate_local_transform (scene/transform.rs:421-540), expression by expression (Rust's
// a + b - c ... is left-associative; x - y is x + (-y)).  One thread per changed node.
// ROT_ONLY: the payload is just the new rotation (16 B); position and scale come from the device-resident copy of
// the node's last full record (trs_by_slot), which every call keeps up to date — property-level change tracking:
// skeletal animation mostly rewrites rotations (Transform::set_rotation), so 20 B per bone cross PCIe instead of 44.
template <bool HAS_STATICS, bool ROT_ONLY>
__global__ void __launch_bounds__(kBlock) k_scatter_trs(const NodeArrays a, const uint32_t count, const uint32_t *d_idx,
                                                        const void *d_payload, fyx_trs *trs_by_slot,
                                                        const fyx_transform_statics *st_by_slot, const uint32_t *slot_of_node,
                                                        const uint32_t n_nodes, uint32_t *d_err)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= count) return;
    const uint32_t slot = resolve_slot(d_idx, e, slot_of_node, n_nodes);
    if (slot == FYX_NONE) return;
    fyx_trs t;
    if (ROT_ONLY) {
        t = trs_by_slot[slot];
        const float4 q = static_cast<const float4 *>(d_payload)[e];
        t.rotation[0] = q.x; t.rotation[1] = q.y; t.rotation[2] = q.z; t.rotation[3] = q.w;
    } else {
        t = static_cast<const fyx_trs *>(d_payload)[e];
    }
    if (trs_by_slot) trs_by_slot[slot] = t;
    Affine A;
    trs_to_local<HAS_STATICS>(t, HAS_STATICS ? st_by_slot + slot : nullptr, A);
    if (!(finite4(A.r0) & finite4(A.r1) & finite4(A.r2))) {
        atomicOr(d_err, E_NOT_AFFINE);
        return;
    }
    a.L[0][slot] = A.r0;
    a.L[1][slot] = A.r1;
    a.L[2][slot] = A.r2;
    atomicOr(a.flags + slot, F_DIRTY_SELF); // NodeMessageKind::TransformChanged
}

__global__ void __launch_bounds__(kBlock) k_scatter_statics(const NodeArrays a, const uint32_t count, const uint32_t *d_idx,
                                                            const fyx_transform_statics *d_in, fyx_transform_statics *st_by_slot,
                                                            const uint32_t *slot_of_node, const uint32_t n_nodes)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= count) return;
    const uint32_t slot = resolve_slot(d_idx, e, slot_of_node, n_nodes);
    if (slot == FYX_NONE) return;
    st_by_slot[slot] = d_in[e];
}

__global__ void __launch_bounds__(kBlock) k_fill_default_statics(fyx_transform_statics *st, const uint32_t n)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= n) return;
    fyx_transform_statics s;
    s.pre_rotation[0] = s.pre_rotation[1] = s.pre_rotation[2] = 0.f;
    s.pre_rotation[3] = 1.f;
    for (int i = 0; i < 9; ++i) s.post_rotation_matrix[i] = (i % 4 == 0) ? 1.f : 0.f;
    for (int i = 0; i < 3; ++i) s.rotation_offset[i] = s.rotation_pivot[i] = s.scaling_offset[i] = s.scaling_pivot[i] = 0.f;
    st[e] = s;
}

// mode 0: node flags (public input bits except ALIVE are replaced); mode 1: plain column store
__global__ void __launch_bounds__(kBlock) k_scatter_u32(uint32_t *dst_col, const uint32_t count, const uint32_t *d_idx,
                                                        const uint32_t *d_val, const uint32_t *slot_of_node,
                                                        const uint32_t n_nodes, const int mode)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= count) return;
    const uint32_t slot = resolve_slot(d_idx, e, slot_of_node, n_nodes);
    if (slot == FYX_NONE) return;
    if (mode == 0) {
        constexpr uint32_t settable = FYX_NODE_INPUT_MASK & ~FYX_NODE_ALIVE;
        const uint32_t old = dst_col[slot];
        dst_col[slot] = (old & ~settable) | (d_val[e] & settable);
    } else {
        dst_col[slot] = d_val[e];
    }
}

__global__ void __launch_bounds__(kBlock) k_scatter_aabbs(const NodeArrays a, const uint32_t count, const uint32_t *d_idx,
                                                          const float *d_aabb6, const uint32_t *slot_of_node,
                                                          const uint32_t n_nodes)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= count) return;
    const uint32_t slot = resolve_slot(d_idx, e, slot_of_node, n_nodes);
    if (slot == FYX_NONE) return;
    const float *b = d_aabb6 + 6 * (size_t)e;
    a.la[0][slot] = make_float2(b[0], b[3]);
    a.la[1][slot] = make_float2(b[1], b[4]);
    a.la[2][slot] = make_float2(b[2], b[5]);
    atomicOr(a.flags + slot, F_DIRTY_SELF); // world box must be rebuilt
}

__global__ void __launch_bounds__(kBlock) k_gather_globals(const NodeArrays a, const uint32_t count, const uint32_t *d_idx,
                                                           const uint32_t *slot_of_node, const uint32_t n_nodes,
                                                           float *d_out)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= count) return;
    const uint32_t slot = resolve_slot(d_idx, e, slot_of_node, n_nodes);
    Affine Gm = affine_identity();
    if (slot != FYX_NONE) {
        Gm.r0 = a.G[0][slot];
        Gm.r1 = a.G[1][slot];
        Gm.r2 = a.G[2][slot];
    }
    float4 *o = reinterpret_cast<float4 *>(d_out + 16 * (size_t)e);
    o[0] = make_float4(Gm.r0.x, Gm.r1.x, Gm.r2.x, 0.0f);
    o[1] = make_float4(Gm.r0.y, Gm.r1.y, Gm.r2.y, 0.0f);
    o[2] = make_float4(Gm.r0.z, Gm.r1.z, Gm.r2.z, 0.0f);
    o[3] = make_float4(Gm.r0.w, Gm.r1.w, Gm.r2.w, 1.0f);
}

__global__ void __launch_bounds__(kBlock) k_gather_aabbs(const NodeArrays a, const uint32_t count, const uint32_t *d_idx,
                                                         const uint32_t *slot_of_node, const uint32_t n_nodes, float *d_out)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= count) return;
    const uint32_t slot = resolve_slot(d_idx, e, slot_of_node, n_nodes);
    float *o = d_out + 6 * (size_t)e;
    if (slot == FYX_NONE) { // AxisAlignedBoundingBox::default()
        o[0] = o[1] = o[2] = 3.402823466e38f;
        o[3] = o[4] = o[5] = -3.402823466e38f;
        return;
    }
    const float2 x = a.wa[0][slot], y = a.wa[1][slot], z = a.wa[2][slot];
    o[0] = x.x; o[1] = y.x; o[2] = z.x;
    o[3] = x.y; o[4] = y.y; o[5] = z.y;
}

__global__ void __launch_bounds__(kBlock) k_gather_flags(const NodeArrays a, const uint32_t count, const uint32_t *d_idx,
                                                         const uint32_t *slot_of_node, const uint32_t n_nodes,
                                                         uint32_t *d_out)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= count) return;
    const uint32_t slot = resolve_slot(d_idx, e, slot_of_node, n_nodes);
    d_out[e] = (slot == FYX_NONE) ? 0u
                                  : (a.flags[slot] & (FYX_NODE_INPUT_MASK | FYX_NODE_GLOBAL_VISIBILITY |
                                                      FYX_NODE_GLOBAL_ENABLED | FYX_NODE_REACHABLE));
}

// VertexBuffer bytes (scene/mesh/buffer.rs:404-414) → the blocked input layout of k_skin (fyx_internal.h).
// Done once per surface at load.  Vertex v (absolute) = group Q = v/4, element j = v%4 of block Q/32.
__global__ void __launch_bounds__(kBlock) k_deinterleave(const uint32_t n_verts, const uint32_t n_padded,
                                                         const unsigned char *d_bytes, const fyx_vertex_layout l,
                                                         const uint32_t n_bones, float4 *vblk, const uint64_t first_vertex,
                                                         uint32_t *d_err)
{
    const uint32_t v = blockIdx.x * kBlock + threadIdx.x;
    if (v >= n_padded) return;
    float p[3] = {0.f, 0.f, 0.f}, n[3] = {0.f, 0.f, 0.f};
    float w[4] = {0.f, 0.f, 0.f, 0.f};
    uint32_t bi = 0u;
    if (v < n_verts) {
        const unsigned char *vp = d_bytes + (size_t)v * l.stride;
        const float *fp = reinterpret_cast<const float *>(vp + l.position_offset);
        const float *fn = reinterpret_cast<const float *>(vp + l.normal_offset);
        const float *fw = reinterpret_cast<const float *>(vp + l.bone_weights_offset);
        p[0] = fp[0]; p[1] = fp[1]; p[2] = fp[2];
        n[0] = fn[0]; n[1] = fn[1]; n[2] = fn[2];
        w[0] = fw[0]; w[1] = fw[1]; w[2] = fw[2]; w[3] = fw[3];
        bi = *reinterpret_cast<const uint32_t *>(vp + l.bone_indices_offset);
        uint32_t bad = 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (((bi >> (8 * k)) & 0xFFu) >= n_bones) bad = 1u;
        if (bad) { // the reference would panic on the out-of-range index (mesh/mod.rs:515)
            atomicOr(d_err, E_BAD_BONE_INDEX);
            bi = 0u;
            w[0] = w[1] = w[2] = w[3] = 0.f;
        }
        if (!((fabsf(p[0]) <= 3.402823466e38f) & (fabsf(p[1]) <= 3.402823466e38f) & (fabsf(p[2]) <= 3.402823466e38f)))
            atomicOr(d_err, E_NONFINITE_VERTEX);
    }
    const uint64_t av = first_vertex + v;
    const uint64_t Q = av >> 2;
    const uint32_t j = (uint32_t)(av & 3);
    float *blk = reinterpret_cast<float *>(vblk + (Q >> 5) * kVblkStride + (Q & 31)); // row 0, this group's float4
    const size_t rs = 32 * 4; // floats between rows
    blk[0 * rs + j] = p[0]; blk[1 * rs + j] = p[1]; blk[2 * rs + j] = p[2];
    blk[3 * rs + j] = n[0]; blk[4 * rs + j] = n[1]; blk[5 * rs + j] = n[2];
    blk[6 * rs + j] = w[0]; blk[7 * rs + j] = w[1]; blk[8 * rs + j] = w[2]; blk[9 * rs + j] = w[3];
    reinterpret_cast<uint32_t *>(blk)[10 * rs + j] = bi;
}

// The tangent (f32 x4 at tangent_offset; .xyz used, .w the handedness stays with the renderer) of a tangent surface →
// its tangent blocks (fyx_internal.h).  Done once per fyx_set_skinned_tangents.  Vertex u of the surface = group u/4,
// element u%4 of block u/128; the padding vertices up to the next multiple of 4 are zero.
__global__ void __launch_bounds__(kBlock) k_tan_deinterleave(const uint32_t n_verts, const uint32_t n_padded, const unsigned char *d_bytes,
                                                             const uint32_t stride, const uint32_t tangent_offset, float4 *tblk)
{
    const uint32_t u = blockIdx.x * kBlock + threadIdx.x;
    if (u >= n_padded) return;
    float t[3] = {0.f, 0.f, 0.f};
    if (u < n_verts) {
        const float *ft = reinterpret_cast<const float *>(d_bytes + (size_t)u * stride + tangent_offset);
        t[0] = ft[0]; t[1] = ft[1]; t[2] = ft[2];
    }
    const uint32_t Q = u >> 2, j = u & 3u;
    float *blk = reinterpret_cast<float *>(tblk + (size_t)(Q >> 5) * kTblkStride + (Q & 31)); // row 0, this group's float4
    const size_t rs = 32 * 4; // floats between rows
    blk[0 * rs + j] = t[0]; blk[1 * rs + j] = t[1]; blk[2 * rs + j] = t[2];
}

__global__ void __launch_bounds__(kBlock) k_ib_rows(const uint32_t n, const float *d_m16, float4 *r0, float4 *r1, float4 *r2,
                                                    uint32_t *d_err)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= n) return;
    Affine A;
    if (!load_affine_rows(d_m16 + 16 * (size_t)e, A)) {
        atomicOr(d_err, E_NOT_AFFINE);
        A = affine_identity();
    }
    r0[e] = A.r0;
    r1[e] = A.r1;
    r2[e] = A.r2;
}

__global__ void k_or_u32(uint32_t *p, const uint32_t bits) { atomicOr(p, bits); }

__global__ void __launch_bounds__(kBlock) k_permute_words(uint32_t *dst, const uint32_t *src, const uint32_t *map, const uint32_t n,
                                                          const uint32_t words, const PermuteDefault def)
{
    const uint64_t t = (uint64_t)blockIdx.x * kBlock + threadIdx.x;
    if (t >= (uint64_t)n * words) return;
    const uint32_t s = (uint32_t)(t / words), w = (uint32_t)(t % words);
    const uint32_t o = map[s];
    dst[t] = (o != FYX_NONE) ? src[(size_t)o * words + w] : def.w[w];
}

// After the fixed-slot NCCL all-gather of a visible list: rank r's entries sit at pad[r*maxc ..];
// pack them back to back (rank order) so every rank holds one contiguous list per frustum.
__global__ void __launch_bounds__(kBlock) k_compact_gathered(const uint32_t *pad, const uint32_t maxc,
                                                             const uint32_t *counts_all, const int nranks, const int f,
                                                             uint32_t *dst)
{
    const uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x;
    if (!maxc) return;
    const uint32_t r = (uint32_t)(i / maxc), j = (uint32_t)(i % maxc);
    if (r >= (uint32_t)nranks) return;
    if (j >= counts_all[r * FYX_MAX_FRUSTA + f]) return;
    uint32_t off = 0;
    for (uint32_t q = 0; q < r; ++q) off += counts_all[q * FYX_MAX_FRUSTA + f];
    dst[off + j] = pad[(size_t)r * maxc + j];
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static inline unsigned grid_for(uint64_t n) { return (unsigned)((n + kBlock - 1) / kBlock); }

// Cull variant (bit 0: warp-level pre-reject of whole frusta, bit 1: warp-wide compaction).  Default: both for
// multi-frustum calls, compaction only for a single frustum; FYX_CULL_VARIANT=0..3 overrides (A/B measurements).
static int cull_variant(int nf)
{
    static int forced = [] {
        const char *e = getenv("FYX_CULL_VARIANT");
        return (e && *e) ? atoi(e) & 63 : -1;
    }();
    if (forced >= 0) return forced;
    (void)nf;
    return 20; // measured (profiles/README.md, round 2): CTA-wide compaction, no pre-reject, FYX_UPDATE_ALL specialisation, 32 registers
}

// bit 3 of the variant: the level kernels store visible bits, k_compact_vis builds the lists (bit 1 is then meaningless)
bool cull_defers_compaction(int nf) { return (cull_variant(nf) & 8) != 0; }

#define FYX_DISPATCH_VAR(KERNEL, NF, VAR, ...)                                   \
    switch (VAR) {                                                               \
    case 0: launch_pdl(KERNEL<NF, 0>, __VA_ARGS__); break;                       \
    case 1: launch_pdl(KERNEL<NF, 1>, __VA_ARGS__); break;                       \
    case 2: launch_pdl(KERNEL<NF, 2>, __VA_ARGS__); break;                       \
    case 3: launch_pdl(KERNEL<NF, 3>, __VA_ARGS__); break;                       \
    case 4: launch_pdl(KERNEL<NF, 4>, __VA_ARGS__); break;                       \
    case 5: launch_pdl(KERNEL<NF, 5>, __VA_ARGS__); break;                       \
    case 6: launch_pdl(KERNEL<NF, 6>, __VA_ARGS__); break;                       \
    case 7: launch_pdl(KERNEL<NF, 7>, __VA_ARGS__); break;                       \
    case 8: launch_pdl(KERNEL<NF, 8>, __VA_ARGS__); break;                       \
    case 9: launch_pdl(KERNEL<NF, 9>, __VA_ARGS__); break;                       \
    case 12: launch_pdl(KERNEL<NF, 12>, __VA_ARGS__); break;                     \
    case 13: launch_pdl(KERNEL<NF, 13>, __VA_ARGS__); break;                     \
    case 20: launch_pdl(KERNEL<NF, 20>, __VA_ARGS__); break;                     \
    case 21: launch_pdl(KERNEL<NF, 21>, __VA_ARGS__); break;                     \
    case 28: launch_pdl(KERNEL<NF, 28>, __VA_ARGS__); break;                     \
    case 32: launch_pdl(KERNEL<NF, 32>, __VA_ARGS__); break;                     \
    case 34: launch_pdl(KERNEL<NF, 34>, __VA_ARGS__); break;                     \
    case 36: launch_pdl(KERNEL<NF, 36>, __VA_ARGS__); break;                     \
    case 38: launch_pdl(KERNEL<NF, 38>, __VA_ARGS__); break;                     \
    case 52: launch_pdl(KERNEL<NF, 52>, __VA_ARGS__); break;                     \
    default: launch_pdl(KERNEL<NF, 54>, __VA_ARGS__); break;                     \
    }

void launch_update_level(cudaStream_t s, const NodeArrays &a, uint32_t lo, uint32_t hi, bool update_all, const CullParams *cull)
{
    if (hi <= lo) return;
    if (cull) {
        const unsigned g = grid_for(hi - lo);
        const uint32_t ua = update_all ? 1u : 0u;
        int var = (cull_variant(cull->nf) & 3) | ((update_all && (cull_variant(cull->nf) & 4)) ? 4 : 0);
        if (cull_variant(cull->nf) & 8) var = (var & 5) | 8; // deferred compaction: 8, 9, 12, 13
        if ((cull_variant(cull->nf) & 16) && update_all) // 32-register builds: 20 (= 4 | 16), 21 (+ pre-reject), 28 (= 12 | 16)
            var = (cull_variant(cull->nf) & 8) ? 28 : ((cull_variant(cull->nf) & 1) ? 21 : 20);
        if (cull_variant(cull->nf) & 32) // warp-convergent predicate: 32, 34 (+ warp compaction); FYX_UPDATE_ALL: 36, 38, 52, 54
            var = 32 | (cull_variant(cull->nf) & 2) | (update_all ? ((cull_variant(cull->nf) & 16) ? 20 : (cull_variant(cull->nf) & 4)) : 0);
        switch (cull->nf) { // the usual frustum counts get an unrolled cull: camera, CSM cascades, cube faces
        case 1: FYX_DISPATCH_VAR(k_update_level, 1, var, g, kBlock, 0, s, a, lo, hi, ua, *cull); break;
        case 2: FYX_DISPATCH_VAR(k_update_level, 2, var, g, kBlock, 0, s, a, lo, hi, ua, *cull); break;
        case 3: FYX_DISPATCH_VAR(k_update_level, 3, var, g, kBlock, 0, s, a, lo, hi, ua, *cull); break;
        case 4: FYX_DISPATCH_VAR(k_update_level, 4, var, g, kBlock, 0, s, a, lo, hi, ua, *cull); break;
        case 6: FYX_DISPATCH_VAR(k_update_level, 6, var, g, kBlock, 0, s, a, lo, hi, ua, *cull); break;
        default: FYX_DISPATCH_VAR(k_update_level, 0, var, g, kBlock, 0, s, a, lo, hi, ua, *cull); break;
        }
    } else {
        CullParams none;
        none.nf = 0;
        if (update_all && (cull_variant(0) & 16)) launch_pdl(k_update_level<-1, 20>, grid_for(hi - lo), kBlock, 0, s, a, lo, hi, 1u, none);
        else if (update_all && (cull_variant(0) & 4)) launch_pdl(k_update_level<-1, 4>, grid_for(hi - lo), kBlock, 0, s, a, lo, hi, 1u, none);
        else launch_pdl(k_update_level<-1, 0>, grid_for(hi - lo), kBlock, 0, s, a, lo, hi, update_all ? 1u : 0u, none);
    }
}

template <int NFT> static void launch_subforest_t(cudaStream_t s, const NodeArrays &a, const SubforestPlan &sf, bool ua, const CullParams &cp)
{
    const bool defer = NFT >= 0 && cull_defers_compaction(cp.nf);
    if (ua && defer) launch_pdl(k_update_subforest<NFT, true, true>, sf.n_ctas, kBlock, 0, s, a, sf.rng, (int)sf.n_levels, 1u, cp);
    else if (ua) launch_pdl(k_update_subforest<NFT, true, false>, sf.n_ctas, kBlock, 0, s, a, sf.rng, (int)sf.n_levels, 1u, cp);
    else if (defer) launch_pdl(k_update_subforest<NFT, false, true>, sf.n_ctas, kBlock, 0, s, a, sf.rng, (int)sf.n_levels, 0u, cp);
    else launch_pdl(k_update_subforest<NFT, false, false>, sf.n_ctas, kBlock, 0, s, a, sf.rng, (int)sf.n_levels, 0u, cp);
}

void launch_update_subforest(cudaStream_t s, const NodeArrays &a, const SubforestPlan &sf, bool update_all, const CullParams *cull)
{
    if (!sf.n_ctas || !sf.n_levels) return;
    if (!cull) {
        CullParams none;
        none.nf = 0;
        launch_subforest_t<-1>(s, a, sf, update_all, none);
        return;
    }
    switch (cull->nf) {
    case 1: launch_subforest_t<1>(s, a, sf, update_all, *cull); break;
    case 6: launch_subforest_t<6>(s, a, sf, update_all, *cull); break;
    default: launch_subforest_t<0>(s, a, sf, update_all, *cull); break;
    }
}

void launch_compact_vis(cudaStream_t s, const NodeArrays &a, const CullParams &cp)
{
    if (!a.cap || !cp.nf) return;
    launch_pdl(k_compact_vis, grid_for(((uint64_t)a.cap + 7) / 8), kBlock, 0, s, a, cp);
}

// Reflection-probe selection of from_graph (renderer/bundle.rs:918-925): the last ReflectionProbe in pool order whose world box
// contains the observer (AxisAlignedBoundingBox::is_contains_point, inclusive) — atomicMax over (node index + 1) per observer.
__global__ void __launch_bounds__(kBlock) k_select_probes(const NodeArrays a, const LodParams obs, uint32_t *best)
{
    const uint32_t slot = blockIdx.x * kBlock + threadIdx.x;
    if (slot >= a.cap) return;
    const uint32_t nf = a.flags[slot];
    if ((nf & (FYX_NODE_ALIVE | FYX_NODE_REFLECTION_PROBE)) != (FYX_NODE_ALIVE | FYX_NODE_REFLECTION_PROBE)) return;
    const float2 wx = a.wa[0][slot], wy = a.wa[1][slot], wz = a.wa[2][slot];
    const uint32_t gi = a.gidx[slot];
    for (int f = 0; f < obs.nf; ++f) {
        const float px = obs.ox[f], py = obs.oy[f], pz = obs.oz[f];
        if (px >= wx.x && px <= wx.y && py >= wy.x && py <= wy.y && pz >= wz.x && pz <= wz.y) atomicMax(best + f, gi + 1u);
    }
}

void launch_select_probes(cudaStream_t s, const NodeArrays &a, const LodParams &obs, uint32_t *best)
{
    if (!a.cap || !obs.nf) return;
    k_select_probes<<<grid_for(a.cap), kBlock, 0, s>>>(a, obs, best);
}

void launch_cull_lights(cudaStream_t s, const NodeArrays &a, const CullParams &cp, uint32_t *const *d_out_ptrs, uint32_t *counts)
{
    if (!a.cap) return;
    k_cull_lights<<<grid_for(a.cap), kBlock, 0, s>>>(a, cp, d_out_ptrs, counts);
}

template <int NF> static void launch_cull_t(cudaStream_t s, unsigned g, int var, const NodeArrays &a, const CullParams &cp, const uint32_t *lodp, uint32_t lo,
                                            uint32_t hi, uint32_t *prune)
{
    switch (var) {
    case 0: k_cull<NF, 0><<<g, kBlock, 0, s>>>(a, cp, lodp, lo, hi, prune); break;
    case 1: k_cull<NF, 1><<<g, kBlock, 0, s>>>(a, cp, lodp, lo, hi, prune); break;
    case 2: k_cull<NF, 2><<<g, kBlock, 0, s>>>(a, cp, lodp, lo, hi, prune); break;
    case 3: k_cull<NF, 3><<<g, kBlock, 0, s>>>(a, cp, lodp, lo, hi, prune); break;
    case 32: k_cull<NF, 32><<<g, kBlock, 0, s>>>(a, cp, lodp, lo, hi, prune); break;
    default: k_cull<NF, 34><<<g, kBlock, 0, s>>>(a, cp, lodp, lo, hi, prune); break;
    }
}

void launch_cull_range(cudaStream_t s, const NodeArrays &a, const CullParams &cp, const uint32_t *lodp, uint32_t lo, uint32_t hi, uint32_t *prune)
{
    if (hi <= lo) return;
    const unsigned g = grid_for(hi - lo);
    const int var = (cull_variant(cp.nf) & 32) ? (32 | (cull_variant(cp.nf) & 2)) : (cull_variant(cp.nf) & 3);
    switch (cp.nf) {
    case 1: launch_cull_t<1>(s, g, var, a, cp, lodp, lo, hi, prune); break;
    case 2: launch_cull_t<2>(s, g, var, a, cp, lodp, lo, hi, prune); break;
    case 3: launch_cull_t<3>(s, g, var, a, cp, lodp, lo, hi, prune); break;
    case 4: launch_cull_t<4>(s, g, var, a, cp, lodp, lo, hi, prune); break;
    case 6: launch_cull_t<6>(s, g, var, a, cp, lodp, lo, hi, prune); break;
    default: launch_cull_t<0>(s, g, var, a, cp, lodp, lo, hi, prune); break;
    }
}

void launch_cull(cudaStream_t s, const NodeArrays &a, const CullParams &cp, const uint32_t *lodp) { launch_cull_range(s, a, cp, lodp, 0u, a.cap, nullptr); }

void launch_fold_bones(cudaStream_t s, const NodeArrays &a, const FoldArrays &fa, const CullParams *cull)
{
    if (!fa.n) return;
    const unsigned grid = grid_for((uint64_t)fa.n * 32); // one warp per skinned mesh
    if (cull) {
        switch (cull->nf) {
        case 1: launch_pdl(k_fold_bones<1>, grid, kBlock, 0, s, a, fa, *cull); break;
        case 6: launch_pdl(k_fold_bones<6>, grid, kBlock, 0, s, a, fa, *cull); break;
        default: launch_pdl(k_fold_bones<0>, grid, kBlock, 0, s, a, fa, *cull); break;
        }
    } else {
        CullParams none;
        none.nf = 0;
        launch_pdl(k_fold_bones<-1>, grid, kBlock, 0, s, a, fa, none);
    }
}

void launch_snapshot_bones(cudaStream_t s, const NodeArrays &a, uint32_t n_late, const uint32_t *late_slot, float4 *stale_pos)
{
    if (!n_late) return;
    k_snapshot_bones<<<grid_for(n_late), kBlock, 0, s>>>(a, n_late, late_slot, stale_pos);
}

void launch_palette(cudaStream_t s, const NodeArrays &a, const SkinArrays &sk)
{
    if (!sk.n_entries) return;
    launch_pdl(k_palette, grid_for(sk.n_entries), kBlock, 0, s, a, sk);
}

template <int S, int LOG2C, int MINB, bool BS, bool TAN> static void launch_skin_t2(cudaStream_t s, const SkinArrays &sk, const SkinTile *tiles, uint32_t n_tiles)
{
    constexpr size_t smem_pal = (size_t)3 * S * (1 << LOG2C) * sizeof(float4);
    static bool init = false;
    if (!init) {
        cudaFuncSetAttribute(k_skin<S, LOG2C, MINB, BS, TAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pal);
        init = true;
    }
    launch_pdl(k_skin<S, LOG2C, MINB, BS, TAN>, n_tiles, kBlock, smem_pal, s, sk, tiles, n_tiles, 1.0f, -0.0f);
}
// CTAs per SM the tangent instantiations are compiled for: 12 more inputs and 12 more accumulators per thread.  At 3 CTAs/SM
// (80 registers) ptxas spills 104-128 B per thread; at 2 (116-124 registers) nothing.
constexpr int kSkinTanMinB = 2;
template <int S, int LOG2C, int MINB, int MINB_TAN>
static void launch_skin_t(cudaStream_t s, const SkinArrays &sk, const SkinTile *tiles, uint32_t n_tiles, bool bs, bool tan)
{
    if (tan) {
        if (bs) launch_skin_t2<S, LOG2C, MINB_TAN, true, true>(s, sk, tiles, n_tiles);
        else launch_skin_t2<S, LOG2C, MINB_TAN, false, true>(s, sk, tiles, n_tiles);
    } else {
        if (bs) launch_skin_t2<S, LOG2C, MINB, true, false>(s, sk, tiles, n_tiles);
        else launch_skin_t2<S, LOG2C, MINB, false, false>(s, sk, tiles, n_tiles);
    }
}

template <int S, int LOG2C, int STAGES, int MINB> static void launch_skin_tma_t(cudaStream_t s, const SkinArrays &sk, const SkinTile *tiles, uint32_t n_tiles)
{
    constexpr size_t pal = ((size_t)3 * S * (1 << LOG2C) * sizeof(float4) + 127) & ~size_t(127);
    constexpr size_t smem = pal + (size_t)(kBlock / 32) * STAGES * kVblkBytes + (size_t)(kBlock / 32) * STAGES * 8;
    static bool init = false;
    if (!init) {
        cudaFuncSetAttribute(k_skin_tma<S, LOG2C, STAGES, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        init = true;
    }
    launch_pdl(k_skin_tma<S, LOG2C, STAGES, MINB>, n_tiles, kBlock, smem, s, sk, tiles, n_tiles, 1.0f, -0.0f);
}

template <int S, int LOG2C, int MINB> static void launch_skin2_t(cudaStream_t s, const SkinArrays &sk, const SkinTile *tiles, uint32_t n_tiles)
{
    constexpr size_t smem_pal = (size_t)3 * S * (1 << LOG2C) * sizeof(float4);
    static bool init = false;
    if (!init) {
        cudaFuncSetAttribute(k_skin2<S, LOG2C, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pal);
        init = true;
    }
    launch_pdl(k_skin2<S, LOG2C, MINB>, n_tiles, kBlock, smem_pal, s, sk, tiles, n_tiles, 1.0f, -0.0f);
}

// 0 = LDG straight into registers (default), 2 = TMA bulk ring (2 stages, 4 palette copies, 2 CTAs/SM), 3 = (3 stages, 8 copies, 1 CTA/SM)
static int skin_variant()
{
    static int v = [] {
        const char *e = getenv("FYX_SKIN_VARIANT");
        if (!e || !*e) return 0;
        if (!strcmp(e, "tma2")) return 2;
        if (!strcmp(e, "tma3")) return 3;
        if (!strcmp(e, "pair4")) return 14; // two vertices per thread, compiled for 4 / 5 / 6 CTAs per SM
        if (!strcmp(e, "pair5")) return 15;
        if (!strcmp(e, "pair6")) return 16;
        return 0;
    }();
    return v;
}

void launch_skin(cudaStream_t s, const SkinArrays &sk, const SkinTile *tiles, uint32_t n_tiles, uint32_t max_bones, bool blend_shapes, bool tangents)
{
    if (!n_tiles) return;
    const int var = skin_variant();
    if (var && max_bones <= 64 && !blend_shapes && !tangents) { // the experiments cover the benchmarked palette size
        if (var == 2) launch_skin_tma_t<65, 2, 2, 2>(s, sk, tiles, n_tiles);
        else if (var == 3) launch_skin_tma_t<65, 3, 3, 1>(s, sk, tiles, n_tiles);
        else if (var == 14) launch_skin2_t<65, 3, 4>(s, sk, tiles, n_tiles);
        else if (var == 15) launch_skin2_t<65, 3, 5>(s, sk, tiles, n_tiles);
        else launch_skin2_t<65, 3, 6>(s, sk, tiles, n_tiles);
        return;
    }
    // 3 CTAs/SM (<= 85 registers): capping at 64 registers for 4 CTAs/SM spills and measured 28 % slower
    if (max_bones <= 64) {       // 8 copies: 25 KB of palette planes
        launch_skin_t<65, 3, 3, kSkinTanMinB>(s, sk, tiles, n_tiles, blend_shapes, tangents);
    } else if (max_bones <= 128) { // 8 copies: 50 KB
        launch_skin_t<129, 3, 3, kSkinTanMinB>(s, sk, tiles, n_tiles, blend_shapes, tangents);
    } else {                       // 4 copies (2-way worst case): 49 KB
        launch_skin_t<257, 2, 3, kSkinTanMinB>(s, sk, tiles, n_tiles, blend_shapes, tangents);
    }
}

void launch_scatter_locals(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx, const float *d_m16,
                           const uint32_t *slot_of_node, uint32_t n_nodes, uint32_t *d_err)
{
    if (!count) return;
    k_scatter_locals<<<grid_for(count), kBlock, 0, s>>>(a, count, d_idx, d_m16, slot_of_node, n_nodes, d_err);
}

void launch_scatter_trs(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx, const void *d_payload, bool rot_only,
                        fyx_trs *trs_by_slot, const fyx_transform_statics *st, const uint32_t *slot_of_node, uint32_t n_nodes,
                        uint32_t *d_err)
{
    if (!count) return;
    const unsigned g = grid_for(count);
    if (rot_only) {
        if (st) k_scatter_trs<true, true><<<g, kBlock, 0, s>>>(a, count, d_idx, d_payload, trs_by_slot, st, slot_of_node, n_nodes, d_err);
        else k_scatter_trs<false, true><<<g, kBlock, 0, s>>>(a, count, d_idx, d_payload, trs_by_slot, st, slot_of_node, n_nodes, d_err);
    } else {
        if (st) k_scatter_trs<true, false><<<g, kBlock, 0, s>>>(a, count, d_idx, d_payload, trs_by_slot, st, slot_of_node, n_nodes, d_err);
        else k_scatter_trs<false, false><<<g, kBlock, 0, s>>>(a, count, d_idx, d_payload, trs_by_slot, st, slot_of_node, n_nodes, d_err);
    }
}

__global__ void __launch_bounds__(kBlock) k_fill_identity_trs(fyx_trs *t, const uint32_t n)
{
    const uint32_t e = blockIdx.x * kBlock + threadIdx.x;
    if (e >= n) return;
    fyx_trs r;
    r.position[0] = r.position[1] = r.position[2] = 0.f;
    r.rotation[0] = r.rotation[1] = r.rotation[2] = 0.f;
    r.rotation[3] = 1.f;
    r.scale[0] = r.scale[1] = r.scale[2] = 1.f;
    t[e] = r;
}

void launch_fill_identity_trs(cudaStream_t s, fyx_trs *t, uint32_t n)
{
    if (!n) return;
    k_fill_identity_trs<<<grid_for(n), kBlock, 0, s>>>(t, n);
}

void launch_scatter_statics(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx, const fyx_transform_statics *d_in,
                            fyx_transform_statics *st, const uint32_t *slot_of_node, uint32_t n_nodes)
{
    if (!count) return;
    k_scatter_statics<<<grid_for(count), kBlock, 0, s>>>(a, count, d_idx, d_in, st, slot_of_node, n_nodes);
}

void launch_fill_default_statics(cudaStream_t s, fyx_transform_statics *st, uint32_t n)
{
    if (!n) return;
    k_fill_default_statics<<<grid_for(n), kBlock, 0, s>>>(st, n);
}

void launch_scatter_u32(cudaStream_t s, uint32_t *dst_col, uint32_t count, const uint32_t *d_idx,
                        const uint32_t *d_val, const uint32_t *slot_of_node, uint32_t n_nodes, int mode)
{
    if (!count) return;
    k_scatter_u32<<<grid_for(count), kBlock, 0, s>>>(dst_col, count, d_idx, d_val, slot_of_node, n_nodes, mode);
}

void launch_scatter_aabbs(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx, const float *d_aabb6,
                          const uint32_t *slot_of_node, uint32_t n_nodes)
{
    if (!count) return;
    k_scatter_aabbs<<<grid_for(count), kBlock, 0, s>>>(a, count, d_idx, d_aabb6, slot_of_node, n_nodes);
}

void launch_gather_globals(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                           const uint32_t *slot_of_node, uint32_t n_nodes, float *d_out)
{
    if (!count) return;
    k_gather_globals<<<grid_for(count), kBlock, 0, s>>>(a, count, d_idx, slot_of_node, n_nodes, d_out);
}

void launch_gather_aabbs(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                         const uint32_t *slot_of_node, uint32_t n_nodes, float *d_out6)
{
    if (!count) return;
    k_gather_aabbs<<<grid_for(count), kBlock, 0, s>>>(a, count, d_idx, slot_of_node, n_nodes, d_out6);
}

void launch_gather_flags(cudaStream_t s, const NodeArrays &a, uint32_t count, const uint32_t *d_idx,
                         const uint32_t *slot_of_node, uint32_t n_nodes, uint32_t *d_out)
{
    if (!count) return;
    k_gather_flags<<<grid_for(count), kBlock, 0, s>>>(a, count, d_idx, slot_of_node, n_nodes, d_out);
}

void launch_deinterleave(cudaStream_t s, uint32_t n_verts, const unsigned char *d_bytes, fyx_vertex_layout layout,
                         uint32_t n_bones, float4 *vblk, uint64_t first_vertex, uint32_t *d_err)
{
    const uint32_t n_padded = (n_verts + 3u) & ~3u;
    if (!n_padded) return;
    k_deinterleave<<<grid_for(n_padded), kBlock, 0, s>>>(n_verts, n_padded, d_bytes, layout, n_bones, vblk, first_vertex, d_err);
}

void launch_tan_deinterleave(cudaStream_t s, uint32_t n_verts, const unsigned char *d_bytes, uint32_t stride, uint32_t tangent_offset, float4 *tblk)
{
    const uint32_t n_padded = (n_verts + 3u) & ~3u;
    if (!n_padded) return;
    k_tan_deinterleave<<<grid_for(n_padded), kBlock, 0, s>>>(n_verts, n_padded, d_bytes, stride, tangent_offset, tblk);
}

void launch_ib_rows(cudaStream_t s, uint32_t n, const float *d_m16, float4 *r0, float4 *r1, float4 *r2, uint32_t *d_err)
{
    if (!n) return;
    k_ib_rows<<<grid_for(n), kBlock, 0, s>>>(n, d_m16, r0, r1, r2, d_err);
}

void launch_or_u32(cudaStream_t s, uint32_t *p, uint32_t bits) { k_or_u32<<<1, 1, 0, s>>>(p, bits); }

void launch_permute_words(cudaStream_t s, void *dst, const void *src, const uint32_t *map, uint32_t n, uint32_t words, const PermuteDefault &def)
{
    if (!n || !words) return;
    k_permute_words<<<grid_for((uint64_t)n * words), kBlock, 0, s>>>(static_cast<uint32_t *>(dst), static_cast<const uint32_t *>(src), map, n, words, def);
}

void launch_compact_gathered(cudaStream_t s, const uint32_t *pad, uint32_t maxc, const uint32_t *counts_all, int nranks, int f,
                             uint32_t *dst)
{
    if (!maxc || nranks <= 0) return;
    k_compact_gathered<<<grid_for((uint64_t)maxc * nranks), kBlock, 0, s>>>(pad, maxc, counts_all, nranks, f, dst);
}

} // namespace fyx
