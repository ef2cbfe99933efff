"""Input shapes at which the kernels switch launch plans: the palette-size bucket of k_skin (<= 64, 65-128, 129-255 bones),
surfaces split into several skinning tiles (more than 8 192 vertices, tiles starting in the middle of a 128-vertex block),
bundle-id spaces wider than the 1 024-entry chunks of k_inst_scan, every frustum count of the fused update + cull + bone fold,
and sub-forest groups filled to exactly kSfCap (384) nodes per level.  Bit for bit against the oracle; the skinning also
against an fp64 linear-blend reference that shares no code with either."""
import ctypes as C

import numpy as np
import pytest

import fyrox_b200 as fb
import oracle_binding as ob
from fyrox_b200.scenegen import Scene
from helpers import NONE, UNIT_BOX, assert_same_hierarchy, assert_same_visible, random_graph, scene_pair
from test_gpu_drawprep import check_instances, observer
from test_gpu_fuzz import random_frusta

pytestmark = pytest.mark.gpu

EYE16 = np.eye(4, dtype=np.float32).reshape(16)
SF_CAP = 384  # kSfCap (fyx_internal.h)


def random_affine(rng, n, spread=4.0):
    """n column-major affine matrices (rotation * scale, translation) with the exact (0, 0, 0, 1) bottom row."""
    out = np.zeros((n, 16), np.float32)
    for i in range(n):
        q, r = np.linalg.qr(rng.normal(size=(3, 3)))
        rot = q * np.sign(np.diag(r))
        m = rot * rng.uniform(0.6, 1.5, 3)  # scale the columns
        out[i, 0:3], out[i, 4:7], out[i, 8:11] = m[:, 0], m[:, 1], m[:, 2]
        out[i, 12:15] = rng.uniform(-spread, spread, 3)
        out[i, 15] = 1.0
    return out


def animated_vertices(rng, nv, nb):
    """Hand-built 68-byte ANIMATED_VERTEX records: bones 0 and nb-1, repeated indices, zero weights."""
    rec = np.zeros((nv, 68), np.uint8)
    f = rec[:, :64].view(np.float32)
    f[:, 0:3] = rng.uniform(-3, 3, (nv, 3))
    f[:, 5:8] = rng.normal(size=(nv, 3))
    w = rng.random((nv, 4)).astype(np.float32)
    w[::3, 2:] = 0.0
    w[1::7, 1:] = 0.0
    f[:, 12:16] = w / w.sum(axis=1, keepdims=True)
    bi = rng.integers(0, nb, (nv, 4)).astype(np.uint8)
    bi[::5] = bi[::5, :1]  # all four influences on one bone
    bi[2::11, 1] = bi[2::11, 3]  # two of four on the same bone
    bi[0] = [0, nb - 1, nb - 1, 0]
    if nv > 1:
        bi[-1] = [nb - 1, 0, nb // 2, nb - 1]
    rec[:, 64:68] = bi
    return rec


def lbs_fp64(pal, rec):
    """Linear-blend skinning in float64 from a palette (n_bones, 16 column-major) and the vertex records, with the per-component
    error bound 2^-20 * sum_k w_k (sum_j |m_ij| |x_j| + |m_i3|) of an fp32 evaluation."""
    f = rec[:, :64].view(np.float32).astype(np.float64)
    p, n, w = f[:, 0:3], f[:, 5:8], f[:, 12:16]
    bi = rec[:, 64:68].astype(np.int64)
    M = pal.astype(np.float64).reshape(-1, 4, 4).transpose(0, 2, 1)[bi]  # (nv, 4, 4, 4): row-major per influence
    R, t = M[..., :3, :3], M[..., :3, 3]
    pos = np.einsum("vk,vkij,vj->vi", w, R, p) + np.einsum("vk,vki->vi", w, t)
    nrm = np.einsum("vk,vkij,vj->vi", w, R, n)
    tol_p = 2.0 ** -20 * (np.einsum("vk,vkij,vj->vi", w, np.abs(R), np.abs(p)) + np.einsum("vk,vki->vi", w, np.abs(t)))
    tol_n = 2.0 ** -20 * np.einsum("vk,vkij,vj->vi", w, np.abs(R), np.abs(n))
    return pos, nrm, tol_p, tol_n


def tiles_of(nv):
    """(tile count, quads per tile) commit_surfaces makes of an nv-vertex surface."""
    quads = (nv + 3) // 4
    nt = (quads + 2047) // 2048
    return nt, (quads + nt - 1) // nt


def skinned_rig(rng, nb, surfaces):
    """A root, nb bones (a random hierarchy under the root) and one mesh node per surface.  surfaces = [(n_bones, n_verts)].
    Each surface gets its own permutation of the bone nodes.  Returns (oracle graph, context loader, per-surface data)."""
    n_surf = len(surfaces)
    n = 1 + nb + n_surf
    parent = np.full(n, NONE, np.uint32)
    parent[1] = 0
    for k in range(2, nb + 1):
        parent[k] = rng.integers(0, k)  # the root or an earlier bone
    parent[nb + 1:] = 0
    flags = np.full(n, fb.NODE_DEFAULT, np.uint32)
    flags[nb + 1:] |= fb.NODE_RENDERABLE
    local = random_affine(rng, n)
    local[0] = EYE16
    ib = random_affine(rng, n, spread=1.0)  # inverse bind pose per bone node
    og = ob.Graph.build(parent, flags, None, local, None)
    for b in range(1, nb + 1):
        og.set_inv_bind(b, ib[b])
    data = []
    for s, (sb, nv) in enumerate(surfaces):
        bones = (1 + rng.permutation(nb)[:sb]).astype(np.uint32)
        rec = animated_vertices(rng, nv, sb)
        og.add_surface(nb + 1 + s, bones, rec.reshape(-1))
        data.append((nb + 1 + s, bones, rec))
    og.L.orc_graph_drop_messages(og.h)
    og.update_hierarchical_data()

    def load(ctx):
        ctx.set_topology(parent, flags)
        ctx.set_local_matrices(local)
        return [ctx.add_skinned_surface(mesh, bones, ib[bones], rec.reshape(-1)) for mesh, bones, rec in data]

    return og, load, data


def check_skinned(og, ctx, sids, data, fp64=True):
    for sid, (mesh, bones, rec) in zip(sids, data):
        nv = rec.shape[0]
        pal_g = ctx.get_palette(sid)
        assert pal_g.tobytes() == og.bone_matrices(mesh, 0, bones.size).tobytes(), f"palette of surface {sid} ({bones.size} bones)"
        pos_g, nrm_g = ctx.get_skinned(sid)
        pos_o, nrm_o = og.skin(mesh, 0, nv)
        bad = np.nonzero((pos_g != pos_o).any(axis=1) | (nrm_g != nrm_o).any(axis=1))[0]
        assert bad.size == 0, f"surface {sid} ({nv} vertices, {bones.size} bones): first differing vertices {bad[:8]}"
        if fp64:
            pos, nrm, tp, tn = lbs_fp64(pal_g, rec)
            ep, en = np.abs(pos_g - pos), np.abs(nrm_g - nrm)
            assert (ep <= tp).all(), f"surface {sid}: position off the fp64 reference by {ep.max()} at vertex {np.argmax((ep - tp).max(axis=1))}"
            assert (en <= tn).all(), f"surface {sid}: normal off the fp64 reference by {en.max()} at vertex {np.argmax((en - tn).max(axis=1))}"


VERT_COUNTS = [1, 5, 127, 128, 129, 8191, 8192, 8193, 12345, 40001]


@pytest.mark.parametrize("nb", [1, 64, 65, 128, 129, 255])
def test_skin_palette_buckets_and_multi_tile_surfaces(ctx, nb):
    """The context's largest bone count picks k_skin<65|129|257, ...>: one context per bucket edge.  Ten surfaces back to back
    (1 ... 40 001 vertices): each starts at a multiple of 4 that is mostly not one of 128, the long ones are cut into 2-5 tiles of
    ceil(quads / tiles) quads that start in the middle of a vertex block."""
    rng = np.random.default_rng(100 + nb)
    surfaces = [(nb if s % 3 != 1 else max(1, nb // 3), nv) for s, nv in enumerate(VERT_COUNTS)]
    og, load, data = skinned_rig(rng, nb, surfaces)
    sids = load(ctx)
    offs = np.cumsum([0] + [(nv + 3) // 4 * 4 for _, nv in surfaces])[:-1]
    assert max(b for b, _ in surfaces) == nb
    assert (offs % 128 != 0).sum() >= 7  # vert_off: surfaces start off the 128-vertex blocks
    assert [tiles_of(nv)[0] for _, nv in surfaces] == [1, 1, 1, 1, 1, 1, 1, 2, 2, 5]
    ctx.update_transforms(fb.UPDATE_ALL)
    ctx.build_palettes()
    ctx.skin()
    check_skinned(og, ctx, sids, data)


def blend_records(rng, ns, stride):
    off = (rng.normal(size=(ns, stride, 9)) * 0.2).astype(np.float16)
    off[rng.random((ns, stride, 9)) < 0.5] = 0
    w = rng.uniform(5, 100, ns).astype(np.float32)
    return off.view(np.uint16), w


@pytest.mark.parametrize("nb", [128, 129])
def test_skin_blend_shapes_on_multi_tile_surfaces(ctx, nb):
    """k_skin<129|257, ..., BS=true>: blend-shape offsets of tiles after the first are found through the tile's local_quad0.
    A 20 000-vertex surface (3 tiles of 1 667 / 1 667 / 1 666 quads) with 3 shapes and layer_stride > n_verts, behind a
    5-vertex surface so that it starts mid-block, and an 8 193-vertex surface (2 tiles) with one shape."""
    rng = np.random.default_rng(200 + nb)
    surfaces = [(nb, 5), (nb, 20000), (max(1, nb - 40), 8193)]
    og, load, data = skinned_rig(rng, nb, surfaces)
    sids = load(ctx)
    assert tiles_of(20000) == (3, 1667) and tiles_of(8193) == (2, 1025)
    shapes = {1: blend_records(rng, 3, 20000 + 77), 2: blend_records(rng, 1, 8193 + 3)}
    for s, (rec, w) in shapes.items():
        ctx.set_blend_shapes(sids[s], rec, w)
    ctx.update_transforms(fb.UPDATE_ALL)
    ctx.build_palettes()
    ctx.skin()
    check_skinned(og, ctx, sids[:1], data[:1])
    L = ob.lib()
    for s, (brec, w) in shapes.items():
        mesh, bones, rec = data[s]
        nv = rec.shape[0]
        pal_o = og.bone_matrices(mesh, 0, bones.size)
        assert ctx.get_palette(sids[s]).tobytes() == pal_o.tobytes()
        pos_o = np.empty((nv, 3), np.float32)
        nrm_o = np.empty((nv, 3), np.float32)
        w100 = (w / np.float32(100.0)).astype(np.float32)
        L.orc_skin_vertices_blend(ob.fp(np.ascontiguousarray(pal_o.reshape(-1))), nv, rec.ctypes.data_as(C.c_void_p), C.byref(ob.ANIMATED_VERTEX), brec.shape[0],
                                  brec.ctypes.data_as(C.c_void_p), brec.shape[1], ob.fp(w100), ob.fp(pos_o.reshape(-1)), ob.fp(nrm_o.reshape(-1)))
        pos_g, nrm_g = ctx.get_skinned(sids[s])
        bad = np.nonzero((pos_g != pos_o).any(axis=1) | (nrm_g != nrm_o).any(axis=1))[0]
        assert bad.size == 0, f"surface {s} ({nv} vertices): first differing vertices {bad[:8]} (tile of {bad[0] // 4 // tiles_of(nv)[1] if bad.size else 0})"
        base = og.skin(mesh, 0, nv)[0]
        assert (pos_g != base).any(axis=1).sum() > nv // 4  # the shapes really moved the later tiles too


@pytest.mark.parametrize("nb", [17, 64])
def test_skin_variant_path_on_multi_tile_surfaces(ctx, nb):
    """The only context shape FYX_SKIN_VARIANT changes (every bone count <= 64, no blend shape): tiles that share a vertex block
    (k_skin_tma's b0 / b1 / q_lo / q_hi, k_skin2's vertex pairs), surfaces of 1 to 40 001 vertices back to back."""
    rng = np.random.default_rng(300 + nb)
    surfaces = [(nb, 3), (nb, 8193), (max(1, nb // 2), 129), (nb, 40001), (nb, 12345), (nb, 8192), (1, 61)]
    assert max(b for b, _ in surfaces) <= 64  # above 64 bones every variant falls back to k_skin
    og, load, data = skinned_rig(rng, nb, surfaces)
    sids = load(ctx)  # and no set_blend_shapes: a shape anywhere in the context also falls back
    ctx.update_transforms(fb.UPDATE_ALL)
    ctx.build_palettes()
    ctx.skin()
    check_skinned(og, ctx, sids, data)
    # a second frame with other bone transforms through the one-call path
    m = random_affine(rng, nb)
    for k in range(nb):
        og.set_local_matrix(1 + k, m[k])
    og.update_hierarchical_data()
    ctx.render_prep(update_flags=fb.UPDATE_ALL, changed_m16=m, changed_idx=np.arange(1, nb + 1, dtype=np.uint32), frusta=[])
    check_skinned(og, ctx, sids, data, fp64=False)


# ---- instance packing over wide bundle-id spaces -----------------------------------------------------------------------
def bundle_pool(n_ids):
    """Bundle ids on both sides of every 1 024-id chunk edge below n_ids, plus 0 and n_ids - 1."""
    pool = {0, 1, n_ids - 1, n_ids - 2}
    for e in range(1024, n_ids + 1, 1024):
        pool |= {e - 2, e - 1, e, e + 1}
    return np.array(sorted(x for x in pool if 0 <= x < n_ids), np.uint32)


SPARSE_POOL = np.array([0, 3, 1023, 1024, 68607, 68608, 68609, 69631, 69632, 69633, 70000], np.uint32)


@pytest.mark.parametrize("n_ids", [1023, 1024, 1025, 5000, 70001])
def test_instances_with_wide_bundle_id_space(ctx, n_ids):
    """k_inst_scan runs one CTA over the histogram in chunks of 1 024 ids and carries the running instance / bundle counts from
    chunk to chunk.  A few thousand visible instances (several CTAs of k_inst_keys / k_inst_scatter), non-empty bundles on both
    sides of each chunk edge; then some nodes with two or three surfaces of their own bundles."""
    parent, flags, mask, local, aabb = random_graph(np.random.default_rng(1025), 5000, p_orphan=0.01)
    rng = np.random.default_rng(n_ids)
    og = ob.Graph.build(parent, flags, mask, local, aabb)
    og.update_hierarchical_data()
    ctx.set_topology(parent, flags, mask, aabb)
    ctx.set_local_matrices(local)
    pool = SPARSE_POOL if n_ids == 70001 else bundle_pool(n_ids)
    bundle = pool[rng.integers(0, pool.size, len(parent))]
    if n_ids != 70001:  # plus a dense spread over the whole space
        some = rng.random(len(parent)) < 0.5
        bundle[some] = rng.integers(0, n_ids, some.sum()).astype(np.uint32)
    bundle[0] = n_ids - 1  # the root (never visible) fixes the id-space size
    ctx.set_bundle_ids(bundle)
    ctx.enable_instances()
    view, vp, fo, ff = observer((0, 0, 120), (0, 0, 0), zf=600.0, fovy=np.deg2rad(100.0))
    ctx.update_and_cull([ff], fb.UPDATE_ALL)
    n = check_instances(og, ctx, 0, fo, view, vp, bundle)
    assert n > 1000
    ids = np.unique(bundle[ctx.get_visible(0)])
    edges = [e for e in range(1024, n_ids, 1024) if np.isin([e - 1, e], pool).all()]  # every edge of the dense cases, three of the sparse one
    assert len(edges) == {1023: 0, 1024: 0, 1025: 1, 5000: 4, 70001: 3}[n_ids]
    for e in edges:  # non-empty bundles right before and right after the chunk edge
        assert np.isin([e - 1, e], ids).all()
    # several surfaces per node (Mesh::surfaces): 2 or 3 instances of the node, each with its own bundle id from the pool
    vis = og.from_graph(fo)
    nodes = rng.choice(vis, 300, replace=False)
    key = {}
    surfaces = []
    for nd in nodes:
        k = int(rng.integers(2, 4))
        lst = [(int(pool[rng.integers(0, pool.size)]), None) for _ in range(k)]
        surfaces.append(lst)
        for s, (bid, _) in enumerate(lst):
            og.add_surface(int(nd), np.empty(0, np.uint32))
            key[(int(nd), s)] = bid
    ctx.set_node_surfaces(nodes, surfaces)
    ctx.cull([ff])
    inst = ctx.pack_instances(0, view, vp)
    node, surf = inst["node"], inst["surface"]
    multi = {int(nd): len(l) for nd, l in zip(nodes, surfaces)}
    want = {(int(nd), s) for nd in vis for s in range(multi.get(int(nd), 1))}
    got = list(zip(node.tolist(), surf.tolist()))
    assert len(got) == len(set(got)) and set(got) == want
    bid = np.array([key.get((nd, s), int(bundle[nd])) for nd, s in got], np.uint32)
    b = inst["bundles"]
    assert np.array_equal(b["id"], np.unique(bid))
    assert b["first"][0] == 0 and np.array_equal(b["first"][1:], np.cumsum(b["count"])[:-1]) and int(b["count"].sum()) == len(got)
    for row in b:
        sl = slice(int(row["first"]), int(row["first"] + row["count"]))
        assert (bid[sl] == row["id"]).all(), f"an instance sits outside bundle {row['id']}"
        assert int(row["sort_index"]) == og.instance(int(node[sl].min()), view, vp)[0]
    for k in range(len(got)):
        si, w, wvp = og.instance(int(node[k]), view, vp)
        assert int(inst["sort_index"][k]) == si
        assert inst["world"][k].tobytes() == w.tobytes() and inst["wvp"][k].tobytes() == wvp.tobytes()


@pytest.mark.parametrize("nb", [65, 129, 255])
def test_instances_bone_blocks_of_large_palettes(ctx, nb):
    """write_uniforms' 255-matrix block of a skinned instance for palettes of 65, 129 and 255 bones: the bone matrices, then
    zero matrices up to 255 (renderer/bundle.rs:484-496)."""
    sc = Scene(5000, 6, verts_per_unit=16, bones_per_unit=nb)
    og, sids = scene_pair(sc, ctx)
    idx, m = sc.animate(2)
    for i, mm in zip(idx, m):
        og.set_local_matrix(int(i), mm)
    og.update_hierarchical_data()
    ctx.enable_instances()
    view, vp, fo, ff = observer((0, 0, 400), (0, 0, 0), zf=900.0)
    ctx.render_prep(update_flags=fb.UPDATE_ALL, changed_m16=m, changed_idx=idx, frusta=[ff])
    inst = ctx.pack_instances(0, view, vp)
    ctx.pack_bone_matrices(0)
    meshes = {int(sc.unit_mesh_node(u)) for u in range(sc.n_units)}
    L = ob.lib()
    seen = 0
    for k, nd in enumerate(inst["node"]):
        blk = ctx.get_bone_matrix_block(0, k)
        want = np.empty(255 * 16, np.float32)
        has = L.orc_instance_bone_block(og.h, int(nd), ob.fp(want))
        assert bool(has) == (int(nd) in meshes) == (blk is not None)
        if has:
            assert blk.reshape(-1).tobytes() == want.tobytes()
            assert blk[:nb].any(axis=1).all()
            assert not blk[nb:].view(np.uint32).any()  # +0.0 padding
            seen += 1
    assert seen >= 3


# ---- every frustum count, with skinned meshes ---------------------------------------------------------------------------
def aimed_frustum(rng, target):
    """A frustum looking at `target` from a random point 10-40 units away."""
    d = rng.normal(size=3)
    eye = np.asarray(target, np.float64) + d / np.linalg.norm(d) * rng.uniform(10, 40)
    up = (0, 1, 0) if abs(d[1]) < 0.9 * np.linalg.norm(d) else (1, 0, 0)
    vp = ob.mat4_mul(ob.perspective(float(rng.uniform(0.8, 1.8)), float(rng.uniform(0.6, 1.6)), 0.1, 300.0), ob.look_at_rh(tuple(eye), tuple(target), up))
    return ob.frustum_from_vp(vp), fb.frustum_from_view_projection_matrix(vp)


@pytest.mark.parametrize("nf", [1, 2, 3, 4, 5, 6, 7, 8])
def test_cull_every_frustum_count_with_skinned_meshes(ctx, nf):
    """k_update_level / k_cull are compiled for 1, 2, 3, 4, 6 frusta and a generic count, k_update_subforest / k_fold_bones for
    1, 6 and generic.  56 skinned units (k_fold_bones on 7 CTAs), frusta alternately random and aimed at a skinned mesh, camera
    masks and shadow passes, through update_and_cull, render_prep and update_transforms + cull."""
    sc = Scene(12000, n_units=56, verts_per_unit=24)
    og, sids = scene_pair(sc, ctx)
    rng = np.random.default_rng(40 + nf)
    meshes = np.array([sc.unit_mesh_node(u) for u in range(sc.n_units)], np.uint32)
    og.update_hierarchical_data()
    fos, ffs = [], []
    rf_o, rf_f = random_frusta(rng, nf)
    for f in range(nf):
        if f % 2:
            o, g = aimed_frustum(rng, og.global_position(int(meshes[rng.integers(0, meshes.size)])))
        else:
            o, g = rf_o[f], rf_f[f]
        fos.append(o)
        ffs.append(g)
    cam = np.full(nf, 0xFFFFFFFF, np.uint32)
    cam[2::4] = 0x0000FFFF
    pf = np.zeros(nf, np.uint32)
    pf[1::3] = fb.PASS_SHADOW
    for frame, entry in enumerate(("update_and_cull", "render_prep", "cull")):
        idx, m = sc.animate(frame)
        for i, mm in zip(idx, m):
            og.set_local_matrix(int(i), mm)
        og.update_hierarchical_data()
        ctx.set_local_matrices(m, idx)
        if entry == "update_and_cull":
            ctx.update_and_cull(ffs, fb.UPDATE_ALL, cam_mask=cam, pass_flags=pf)
        elif entry == "render_prep":
            ctx.render_prep(update_flags=fb.UPDATE_ALL, frusta=ffs, cam_mask=cam, pass_flags=pf)
        else:
            ctx.update_transforms(fb.UPDATE_ALL)
            ctx.cull(ffs, cam_mask=cam, pass_flags=pf)
        assert_same_hierarchy(og, ctx, meshes)
        for f in range(nf):
            want = np.sort(og.from_graph(fos[f], int(cam[f]), bool(pf[f] & fb.PASS_SHADOW)))
            got = np.sort(ctx.get_visible(f))
            assert np.array_equal(got, want), f"{entry}, frustum {f} of {nf}: {got.size} visible on the GPU, {want.size} in the oracle"
            if f % 2:  # the aimed frusta do see skinned meshes: the fold's own cull decides for them
                assert np.isin(want, meshes).any(), f"frustum {f} sees no skinned mesh"


# ---- sub-forest groups at kSfCap -----------------------------------------------------------------------------------------
def subforest_plan(parent):
    """What the topology upload plans for k_update_subforest (fyx_api.cu), for a tree under node 0 whose nodes come in level
    order: (first level, [per group: node count of each level from that one down]).  The default mode (no FYX_SUBFOREST)."""
    n = len(parent)
    depth = np.zeros(n, np.int64)
    for i in range(1, n):
        depth[i] = depth[parent[i]] + 1
    assert (np.diff(depth) >= 0).all()
    nlev = int(depth.max()) + 1
    size = np.ones(n, np.int64)
    for i in range(n - 1, 0, -1):
        size[parent[i]] += size[i]
    for l in range(1, nlev - 2):
        lv = np.nonzero(depth == l)[0]
        if size[lv].max() <= SF_CAP and (depth >= l).sum() >= 8 * lv.size:
            break
    else:
        return None, []
    top = np.arange(n)
    for i in range(n):
        if depth[i] > l:
            top[i] = top[parent[i]]
    groups, acc = [], np.zeros(nlev - l, np.int64)
    for t in np.nonzero(depth == l)[0]:
        cnt = np.bincount(depth[(top == t) & (depth >= l)] - l, minlength=nlev - l)
        if (acc + cnt > SF_CAP).any():
            groups.append(acc.tolist())
            acc = np.zeros_like(acc)
        acc += cnt
    groups.append(acc.tolist())
    return l, groups


def capacity_forest(rng, last):
    """Under the root: four sub-trees of 1 + 4 + 128 + 128 nodes (three fill a group level to exactly 384, the fourth opens the
    next group), one sub-tree of `last` = 384 or 385 nodes (1 + 1 + 382 or 383 in a chain of levels), then 12 leaves."""
    trees = [[1, 4, 128, 128]] * 4 + [[1, 1, last - 2]] + [[1]] * 12
    parent = [NONE]
    members = []  # per tree, per level: its nodes
    for widths in trees:
        members.append([[] for _ in widths])
    for depth in range(4):
        for t, widths in enumerate(trees):
            if depth >= len(widths):
                continue
            for j in range(widths[depth]):
                members[t][depth].append(len(parent))
                if depth == 0:
                    parent.append(0)
                else:
                    up = members[t][depth - 1]
                    parent.append(up[j * len(up) // widths[depth]])
    parent = np.array(parent, np.uint32)
    n = len(parent)
    flags = np.full(n, fb.NODE_DEFAULT | fb.NODE_RENDERABLE, np.uint32)
    flags[0] = fb.NODE_DEFAULT
    flags[rng.random(n) < 0.05] &= ~np.uint32(fb.NODE_VISIBILITY)
    mask = np.where(rng.random(n) < 0.9, 0xFFFFFFFF, 0x0000FFFF).astype(np.uint32)
    local = random_affine(rng, n, spread=3.0)
    local[0] = EYE16
    h = rng.uniform(0.1, 1.5, (n, 3)).astype(np.float32)
    aabb = np.concatenate([-h, h], axis=1)
    aabb[0] = UNIT_BOX  # the root is a pivot: the oracle gives it Base's unit box
    return parent, flags, mask, local, aabb


@pytest.mark.parametrize("last", [384, 385])
def test_cull_subforest_groups_at_capacity(ctx, last):
    """k_update_subforest groups whole sub-trees until a level would pass kSfCap = 384 nodes, from the first level whose sub-trees
    all have <= 384 nodes.  With a 384-node sub-tree level 1 is that level and three sub-trees fill their group's two deepest
    levels to exactly 384; with 385 nodes level 1 is skipped and level 2 is taken, where twelve sub-trees fill a group to 384
    again.  Full and incremental updates, fused and stand-alone culls with 1, 3 and 6 frusta."""
    rng = np.random.default_rng(last)
    parent, flags, mask, local, aabb = capacity_forest(rng, last)
    first, groups = subforest_plan(parent)
    if last == 384:
        assert first == 1 and groups[0] == [3, 12, 384, 384] and groups[1] == [1, 4, 128, 128] and groups[2][2] == 382
    else:
        assert first == 2 and groups[0] == [12, 384, 384] and groups[1] == [4, 128, 128] and groups[2] == [1, 383, 0]
    og = ob.Graph.build(parent, flags, mask, local, aabb)
    og.update_hierarchical_data()
    ctx.set_topology(parent, flags, mask, aabb)
    ctx.set_local_matrices(local)
    n = len(parent)
    seen = 0
    for step, nf in enumerate((1, 3, 6)):
        fos, ffs = random_frusta(rng, nf)
        cam = np.full(nf, 0xFFFFFFFF, np.uint32)
        cam[1::2] = 0xFFFF0000
        if step:  # move some nodes of every level, then an incremental update
            moved = np.sort(rng.choice(np.arange(1, n), 200, replace=False)).astype(np.uint32)
            m = random_affine(rng, moved.size, spread=3.0)
            for i, mm in zip(moved, m):
                og.set_local_matrix(int(i), mm)
            og.update()
            ctx.set_local_matrices(m, moved)
            ctx.update_and_cull(ffs, fb.UPDATE_INCREMENTAL, cam_mask=cam)
        else:
            ctx.update_and_cull(ffs, fb.UPDATE_ALL, cam_mask=cam)
        assert_same_hierarchy(og, ctx)
        assert_same_visible(og, ctx, fos, cam)
        seen += sum(ctx.get_visible(f).size for f in range(nf))
        ctx.update_transforms(fb.UPDATE_ALL)
        ctx.cull(ffs, cam_mask=cam)
        assert_same_hierarchy(og, ctx)
        assert_same_visible(og, ctx, fos, cam)
    assert seen > 100
