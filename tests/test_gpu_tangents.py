"""Skinned tangents (fyx_set_skinned_tangents): the third stream of k_skin<..., TAN = true>.  Every check is bit for bit against
the oracle's normal path pointed at the tangent attribute (test_skin_tangents_cpu.oracle_tangents) and within 2^-20 of a float64
linear blend that shares no code with either.  Surfaces without tangents must come out exactly as in a context that has none."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import fyrox_b200 as fb
from fyrox_b200 import _lib as L
from fyrox_b200.context import FyxError
from helpers import NONE
from test_gpu_shapes import EYE16, blend_records, check_skinned, random_affine, skinned_rig, tiles_of
from test_skin_tangents_cpu import oracle_tangents

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def add_tangents(rng, data, every=1):
    """Random tangents (xyz, handedness +-1 in w) at offset 32 of the records of surfaces 0, every, 2*every, ... (in place)."""
    for s, (_, _, rec) in enumerate(data):
        f = rec[:, :64].view(np.float32)
        f[:, 8:11] = rng.normal(size=(rec.shape[0], 3))
        f[::7, 8] = -0.0
        f[:, 11] = np.where(rng.random(rec.shape[0]) < 0.5, -1.0, 1.0)
    return [s for s in range(len(data)) if s % every == 0]


def tan_fp64(pal, rec):
    f = rec[:, :64].view(np.float32).astype(np.float64)
    t, w = f[:, 8:11], f[:, 12:16]
    R = pal.astype(np.float64).reshape(-1, 4, 4).transpose(0, 2, 1)[rec[:, 64:68].astype(np.int64)][..., :3, :3]
    return np.einsum("vk,vkij,vj->vi", w, R, t), 2.0 ** -20 * np.einsum("vk,vkij,vj->vi", w, np.abs(R), np.abs(t))


def check_tangents(ctx, sid, rec, shapes=None, weights100=None, fp64=True):
    pal = ctx.get_palette(sid)
    got = ctx.get_skinned_tangents(sid)
    want = oracle_tangents(pal, rec, shapes=shapes, weights100=weights100)
    bad = np.nonzero((got.view(np.uint32) != want.view(np.uint32)).any(axis=1))[0]
    nv = rec.shape[0]
    assert bad.size == 0, f"surface {sid} ({nv} vertices): first differing tangents {bad[:8]} (tile {bad[0] // 4 // tiles_of(nv)[1] if bad.size else 0})"
    if fp64 and shapes is None:
        t, tol = tan_fp64(pal, rec)
        err = np.abs(got - t)
        assert (err <= tol).all(), f"surface {sid}: tangent off the fp64 reference by {err.max()}"
    assert ctx.get_skinned_tangents_device(sid)


class Recorder:
    """Passes calls through to a context and remembers the arguments of the last call of each method."""

    def __init__(self, ctx):
        self.ctx, self.calls = ctx, {}

    def __getattr__(self, name):
        f = getattr(self.ctx, name)

        def call(*a, **k):
            self.calls[name] = a
            return f(*a, **k)

        return call


def frame(ctx):
    ctx.update_transforms(fb.UPDATE_ALL)
    ctx.build_palettes()
    ctx.skin()


VERT_COUNTS = [1, 3, 127, 129, 8193, 5, 40001, 12345]


@pytest.mark.parametrize("nb", [1, 64, 65, 128, 129, 255])
def test_tangents_palette_buckets_and_multi_tile_surfaces(ctx, nb):
    """k_skin<65|129|257, 3|2, 2, false, true>: surfaces of 1 ... 40 001 vertices back to back, padding, 2- and 5-tile surfaces
    whose later tiles start in the middle of a 128-vertex block.  Positions and normals stay exact as well."""
    rng = np.random.default_rng(400 + nb)
    surfaces = [(nb if s % 3 != 1 else max(1, nb // 3), nv) for s, nv in enumerate(VERT_COUNTS)]
    og, load, data = skinned_rig(rng, nb, surfaces)
    add_tangents(rng, data)
    sids = load(ctx)
    assert [tiles_of(nv)[0] for _, nv in surfaces] == [1, 1, 1, 1, 2, 1, 5, 2]
    for sid, (_, _, rec) in zip(sids, data):
        ctx.set_skinned_tangents(sid, rec.reshape(-1))
    frame(ctx)
    check_skinned(og, ctx, sids, data)
    for sid, (_, _, rec) in zip(sids, data):
        check_tangents(ctx, sid, rec)


@pytest.mark.parametrize("nb", [64, 129])
def test_mixed_context_leaves_the_other_streams_alone(nb):
    """Tangent surfaces interleaved with tangent-less ones: the positions and normals of EVERY surface are bit-identical to the
    same scene loaded with no tangents at all (which runs the TAN = false kernel), the tangent-less getters say FYX_ERR_STATE."""
    rng = np.random.default_rng(500 + nb)
    surfaces = [(nb, nv) for nv in [3, 8193, 129, 40001, 1, 12345, 640]]
    og, load, data = skinned_rig(rng, nb, surfaces)
    with_tan = add_tangents(rng, data, every=2)
    with fb.Context() as plain, fb.Context() as mixed:
        sp, sm = load(plain), load(mixed)
        for s in with_tan:
            mixed.set_skinned_tangents(sm[s], data[s][2].reshape(-1))
        for c in (plain, mixed):
            frame(c)
        for a, b, (_, _, rec) in zip(sp, sm, data):
            pa, na = plain.get_skinned(a)
            pm, nm = mixed.get_skinned(b)
            assert pa.tobytes() == pm.tobytes() and na.tobytes() == nm.tobytes(), f"surface {b}"
        check_skinned(og, mixed, sm, data, fp64=False)
        for s, (sid, (_, _, rec)) in enumerate(zip(sm, data)):
            if s in with_tan:
                check_tangents(mixed, sid, rec)
            else:
                with pytest.raises(FyxError) as e:
                    mixed.get_skinned_tangents(sid)
                assert e.value.code == L.FYX_ERR_STATE


@pytest.mark.parametrize("nb", [128, 129])
def test_tangent_blend_shapes_on_multi_tile_surfaces(ctx, nb):
    """k_skin<..., BS = true, TAN = true>: the tangent offsets (halfs 6-8) of tiles after the first are found through local_quad0;
    weight updates, shapes removed; fyx_set_skinned_tangents after the shapes is FYX_ERR_STATE."""
    rng = np.random.default_rng(600 + nb)
    surfaces = [(nb, 5), (nb, 20000), (max(1, nb - 40), 8193), (nb, 300)]
    og, load, data = skinned_rig(rng, nb, surfaces)
    add_tangents(rng, data)
    sids = load(ctx)
    assert tiles_of(20000) == (3, 1667) and tiles_of(8193) == (2, 1025)
    for sid, (_, _, rec) in zip(sids, data):
        ctx.set_skinned_tangents(sid, rec.reshape(-1))
    shapes = {1: blend_records(rng, 3, 20000 + 77), 2: blend_records(rng, 1, 8193 + 3)}
    for s, (brec, w) in shapes.items():
        ctx.set_blend_shapes(sids[s], brec.reshape(brec.shape[0], -1, 9), w)
    frame(ctx)
    check_tangents(ctx, sids[0], data[0][2])
    check_tangents(ctx, sids[3], data[3][2])
    for s, (brec, w) in shapes.items():
        check_tangents(ctx, sids[s], data[s][2], brec, w)
        plain = oracle_tangents(ctx.get_palette(sids[s]), data[s][2])
        assert (ctx.get_skinned_tangents(sids[s]) != plain).any(axis=1).sum() > data[s][2].shape[0] // 4  # later tiles moved too
    # weight updates
    w1 = np.array([0.0, 100.0, 12.5], np.float32)
    ctx.set_blend_shape_weights(sids[1], w1)
    frame(ctx)
    check_tangents(ctx, sids[1], data[1][2], shapes[1][0], w1)
    check_tangents(ctx, sids[2], data[2][2], *shapes[2])
    # a surface with shapes cannot turn tangents on (again)
    for args in ((sids[1], data[1][2].reshape(-1)), (sids[2], data[2][2].reshape(-1))):
        with pytest.raises(FyxError) as e:
            ctx.set_skinned_tangents(*args)
        assert e.value.code == L.FYX_ERR_STATE and b"fyx_set_blend_shapes" in L.load().fyx_last_error(ctx._h)
    # shapes removed: the plain tangents again
    ctx.set_blend_shapes(sids[1], np.zeros((0, 0, 9), np.uint16))
    frame(ctx)
    check_tangents(ctx, sids[1], data[1][2])
    check_tangents(ctx, sids[2], data[2][2], *shapes[2])
    # argument checks
    for stride, off in ((68, 30), (68, 56), (66, 32)):  # misaligned offset, tangent past the vertex, misaligned stride
        with pytest.raises(FyxError) as e:
            ctx.set_skinned_tangents(sids[0], data[0][2].reshape(-1), off, stride)
        assert e.value.code == L.FYX_ERR_INVALID_ARGUMENT


def test_k16_reference_vertex_tangent_offset_40(ctx):
    """tests/golden K16: the reference's 76-byte test vertex (tangent f32 x4 at 40).  Bones translate only and the weights are
    0.25 each, so every tangent comes out as its own xyz, exactly; bit for bit the oracle's too."""
    k = json.load(open(os.path.join(HERE, "golden", "reference_kats.json")))["K16_vertex_buffer_attributes"]
    off = k["offsets"]
    nv = len(k["vertices"])
    rec = np.zeros((nv, k["stride"]), np.uint8)
    for i, v in enumerate(k["vertices"]):
        for name in ("position", "tex_coord", "second_tex_coord", "normal", "tangent", "bone_weights"):
            a = np.asarray(v[name], np.float32)
            rec[i, off[name]:off[name] + 4 * a.size] = a.view(np.uint8)
        rec[i, off["bone_indices"]:off["bone_indices"] + 4] = np.asarray(v["bone_indices"], np.uint8)
    nb = 6
    n = nb + 2
    parent = np.array([NONE] + [0] * (n - 1), np.uint32)
    flags = np.full(n, fb.NODE_DEFAULT, np.uint32)
    flags[n - 1] |= fb.NODE_RENDERABLE
    local = np.tile(EYE16, (n, 1))
    for b in range(nb):
        local[1 + b, 12] = float(b)
    ctx.set_topology(parent, flags)
    ctx.set_local_matrices(local)
    layout = L.fyx_vertex_layout(k["stride"], off["position"], off["normal"], off["bone_weights"], off["bone_indices"])
    sid = ctx.add_skinned_surface(n - 1, np.arange(1, nb + 1, dtype=np.uint32), np.tile(EYE16, (nb, 1)), rec.reshape(-1), layout=layout)
    ctx.set_skinned_tangents(sid, rec.reshape(-1), off["tangent"], k["stride"])
    frame(ctx)
    tan = ctx.get_skinned_tangents(sid)
    for i, v in enumerate(k["vertices"]):
        assert np.array_equal(tan[i], np.asarray(v["tangent"][:3], np.float32)), (i, tan[i])
    lay = __import__("oracle_binding").VertexLayout(k["stride"], off["position"], off["normal"], off["bone_weights"], off["bone_indices"])
    assert tan.tobytes() == oracle_tangents(ctx.get_palette(sid), rec, off["tangent"], lay).tobytes()


def test_tangents_through_render_prep_topology_change_and_off(ctx):
    """Several frames of changing bones through fyx_render_prep, synchronous and pipelined (FYX_FRAME_ASYNC); a fyx_set_topology
    change (the tangent data belongs to the surface and stays); tangents turned off again: the getter says FYX_ERR_STATE and the
    positions and normals are unchanged."""
    rng = np.random.default_rng(700)
    nb = 40
    surfaces = [(nb, 8193), (nb // 2, 77), (nb, 3000)]
    og, load, data = skinned_rig(rng, nb, surfaces)
    add_tangents(rng, data)
    rec_ctx = Recorder(ctx)
    sids = load(rec_ctx)
    for sid, (_, _, rec) in zip(sids, data):
        ctx.set_skinned_tangents(sid, rec.reshape(-1))
    bone_idx = np.arange(1, nb + 1, dtype=np.uint32)
    for fr in range(6):
        m = random_affine(rng, nb)
        for k in range(nb):
            og.set_local_matrix(1 + k, m[k])
        og.update_hierarchical_data()
        ctx.render_prep(update_flags=fb.UPDATE_ALL, changed_m16=m, changed_idx=bone_idx, frusta=[], readback_visible=False, async_=fr % 2 == 1)
        ctx.sync()
        check_skinned(og, ctx, sids, data, fp64=False)
        for sid, (_, _, rec) in zip(sids, data):
            check_tangents(ctx, sid, rec, fp64=fr == 0)
    # topology change: one more node under the root; every node keeps its index, the bones their last matrices
    parent, flags = rec_ctx.calls["set_topology"]
    local = rec_ctx.calls["set_local_matrices"][0].copy()
    local[1:nb + 1] = m
    ctx.set_topology(np.append(parent, np.uint32(0)), np.append(flags, np.uint32(fb.NODE_DEFAULT)))
    ctx.set_local_matrices(np.vstack([local, EYE16]))
    ctx.render_prep(update_flags=fb.UPDATE_ALL, frusta=[], readback_visible=False)
    check_skinned(og, ctx, sids, data, fp64=False)
    for sid, (_, _, rec) in zip(sids, data):
        check_tangents(ctx, sid, rec, fp64=False)
    # off again
    before = [ctx.get_skinned(s) for s in sids]
    ctx.set_skinned_tangents(sids[0], None)
    ctx.render_prep(update_flags=fb.UPDATE_ALL, frusta=[], readback_visible=False)
    with pytest.raises(FyxError) as e:
        ctx.get_skinned_tangents(sids[0])
    assert e.value.code == L.FYX_ERR_STATE
    with pytest.raises(FyxError):
        ctx.get_skinned_tangents_device(sids[0])
    for s, (p, nr) in zip(sids, before):
        p2, n2 = ctx.get_skinned(s)
        assert p.tobytes() == p2.tobytes() and nr.tobytes() == n2.tobytes()
    check_tangents(ctx, sids[1], data[1][2], fp64=False)


@pytest.mark.timeout(1000)
@pytest.mark.parametrize("variant", ["tma2", "pair5"])
def test_tangents_under_skin_variants(variant):
    """FYX_SKIN_VARIANT does not cover tangents: a context with a tangent surface takes the default LDG kernel whatever it says."""
    e = dict(os.environ)
    e["FYX_SKIN_VARIANT"] = variant
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-k", "not variants", os.path.join(HERE, "test_gpu_tangents.py")],
                       capture_output=True, text=True, env=e, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
