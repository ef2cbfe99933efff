"""Skinned tangents, CPU side.  The standard shader skins the tangent with the normal's arithmetic (standard.shader:167-173
for the blend shapes, :192-200 for the skinning), so the oracle of the tangent stream is the oracle's normal path
(orc_skin_vertices / orc_skin_vertices_blend) pointed at the tangent attribute: a vertex layout whose normal offset is the
tangent offset, and blend-shape records whose halfs 3-5 carry halfs 6-8.  Checked here against an independent numpy float32
restatement of the op order (random vertices, zero weights, -0, subnormals, every finite binary16 offset), plus the argument
checks of the three entry points, which need no GPU."""
import ctypes as C

import numpy as np

import fyrox_b200._lib as L
import oracle_binding as ob

TANGENT_OFFSET = 32  # AnimatedVertex: position 0, tex 12, normal 20, tangent 32, weights 48, indices 64


def tangent_layout(layout, tangent_offset):
    """The oracle's vertex layout with the normal read from the tangent attribute."""
    return ob.VertexLayout(layout.stride, layout.position_offset, tangent_offset, layout.bone_weights_offset, layout.bone_indices_offset)


def oracle_tangents(pal, rec, tangent_offset=TANGENT_OFFSET, layout=ob.ANIMATED_VERTEX, shapes=None, weights100=None):
    """Skinned tangents (n_verts, 3) of the records `rec` (uint8 (n_verts, stride)) under the palette pal (n_bones, 16);
    shapes = uint16 (n_shapes, layer_stride, 9) blend-shape records with BlendShape::weight values weights100."""
    nv = rec.shape[0]
    lay = tangent_layout(layout, tangent_offset)
    pal = np.ascontiguousarray(pal, np.float32).reshape(-1)
    rec = np.ascontiguousarray(rec)
    pos = np.empty((nv, 3), np.float32)
    tan = np.empty((nv, 3), np.float32)
    L_ = ob.lib()
    if shapes is None or len(shapes) == 0:
        L_.orc_skin_vertices(ob.fp(pal), nv, rec.ctypes.data_as(C.c_void_p), C.byref(lay), ob.fp(pos.reshape(-1)), ob.fp(tan.reshape(-1)))
    else:
        r = np.ascontiguousarray(shapes, np.uint16).copy()
        r[..., 3:6] = r[..., 6:9]  # the tangent offsets where the oracle reads the normal's
        w = (np.asarray(weights100, np.float32) / np.float32(100.0)).astype(np.float32)
        L_.orc_skin_vertices_blend(ob.fp(pal), nv, rec.ctypes.data_as(C.c_void_p), C.byref(lay), r.shape[0], r.ctypes.data_as(C.c_void_p), r.shape[1],
                                   ob.fp(w), ob.fp(pos.reshape(-1)), ob.fp(tan.reshape(-1)))
    return tan


def numpy_tangents(pal, t, w, bi):
    """r_i = (m_i0*tx + m_i1*ty) + m_i2*tz; acc_i += r_i * w_k for k = 0..3, every step one float32 rounding."""
    M = np.asarray(pal, np.float32).reshape(-1, 16)
    acc = np.zeros((t.shape[0], 3), np.float32)
    for k in range(4):
        m = M[bi[:, k]]
        for i in range(3):
            r = (m[:, 0 + i] * t[:, 0] + m[:, 4 + i] * t[:, 1]) + m[:, 8 + i] * t[:, 2]
            acc[:, i] = acc[:, i] + r * w[:, k]
    return acc


def random_records(rng, nv, nb):
    rec = np.zeros((nv, 68), np.uint8)
    f = rec[:, :64].view(np.float32)
    f[:, 0:3] = rng.uniform(-3, 3, (nv, 3))
    f[:, 5:8] = rng.normal(size=(nv, 3))
    f[:, 8:12] = rng.normal(size=(nv, 4))
    f[:, 11] = np.where(rng.random(nv) < 0.5, -1.0, 1.0)  # handedness: never read
    w = rng.random((nv, 4)).astype(np.float32)
    w[::3, 2:] = 0.0  # zero weights
    w[1::7, 1:] = 0.0
    f[:, 12:16] = w / w.sum(axis=1, keepdims=True)
    # -0 and subnormal tangent components
    f[::5, 8] = -0.0
    f[1::6, 9] = np.float32(1e-40)
    f[2::9, 10] = -np.float32(3e-39)
    f[3::13, 8:11] = 0.0
    rec[:, 64:68] = rng.integers(0, nb, (nv, 4)).astype(np.uint8)
    return rec


def random_palette(rng, nb):
    pal = np.zeros((nb, 16), np.float32)
    pal[:, [0, 1, 2, 4, 5, 6, 8, 9, 10]] = rng.normal(size=(nb, 9))
    pal[:, 12:15] = rng.uniform(-4, 4, (nb, 3))
    pal[:, 15] = 1.0
    pal[0, :] = np.eye(4, dtype=np.float32).reshape(16)
    pal[1, 0] = -0.0
    return pal


def test_oracle_tangents_equal_the_numpy_restatement():
    rng = np.random.default_rng(11)
    nv, nb = 5000, 40
    rec = random_records(rng, nv, nb)
    pal = random_palette(rng, nb)
    f = rec[:, :64].view(np.float32)
    got = oracle_tangents(pal, rec)
    want = numpy_tangents(pal, f[:, 8:11].copy(), f[:, 12:16].copy(), rec[:, 64:68].astype(np.int64))
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert (got[f[:, 8:11].any(axis=1) == 0] == 0).all()


def test_tangent_equal_to_the_normal_skins_to_the_oracle_normal():
    """The tangent path is the pinned normal path: fed tangent == normal it returns the oracle's normals bit for bit."""
    rng = np.random.default_rng(12)
    nv, nb = 3000, 255
    rec = random_records(rng, nv, nb)
    rec[:, 32:44] = rec[:, 20:32]
    pal = random_palette(rng, nb)
    pos = np.empty((nv, 3), np.float32)
    nrm = np.empty((nv, 3), np.float32)
    ob.lib().orc_skin_vertices(ob.fp(pal.reshape(-1)), nv, rec.ctypes.data_as(C.c_void_p), C.byref(ob.ANIMATED_VERTEX), ob.fp(pos.reshape(-1)),
                               ob.fp(nrm.reshape(-1)))
    assert np.array_equal(oracle_tangents(pal, rec).view(np.uint32), nrm.view(np.uint32))


def test_blend_shape_tangent_offsets_over_every_finite_half():
    """Halfs 6-8 of every record, in shape order: t += offset.tangent * weight (one rounding per product and sum), over every
    finite binary16 pattern incl. subnormals and both zeros; an identity palette with weights (1, 0, 0, 0) passes it through."""
    rng = np.random.default_rng(13)
    nv, ns = 8192, 3  # 3 x 8 192 x 3 tangent slots that are read hold all 63 488 finite patterns
    pats = np.arange(65536, dtype=np.uint16)
    finite = pats[np.isfinite(pats.view(np.float16))]
    shapes = finite[rng.integers(0, len(finite), (ns, nv + 7, 9))].astype(np.uint16)  # layer_stride = nv + 7 (padding texels)
    tan_slots = shapes[:, :nv, 6:9].reshape(-1)
    tan_slots[: len(finite)] = finite
    shapes[:, :nv, 6:9] = tan_slots.reshape(ns, nv, 3)
    weights100 = np.array([100.0, 37.5, 0.0], np.float32)
    rec = np.zeros((nv, 68), np.uint8)
    f = rec[:, :64].view(np.float32)
    f[:, 8:11] = rng.normal(size=(nv, 3))
    f[:, 12] = 1.0
    pal = np.eye(4, dtype=np.float32).reshape(1, 16)
    with np.errstate(over="ignore", invalid="ignore"):
        got = oracle_tangents(pal, rec, shapes=shapes, weights100=weights100)
        t = f[:, 8:11].copy()
        w = (weights100 / np.float32(100.0)).astype(np.float32)
        for i in range(ns):
            t = t + shapes[i, :nv, 6:9].view(np.float16).astype(np.float32) * w[i]
        want = t + np.float32(0.0)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_tangent_entry_points_reject_a_null_context_without_a_gpu():
    lib = L.load()
    buf = (C.c_float * 12)()
    p = C.c_void_p()
    assert lib.fyx_set_skinned_tangents(None, 0, C.cast(buf, C.c_void_p), 68, 32) == L.FYX_ERR_INVALID_ARGUMENT
    assert lib.fyx_get_skinned_tangents(None, 0, C.cast(buf, C.c_void_p)) == L.FYX_ERR_INVALID_ARGUMENT
    assert lib.fyx_get_skinned_tangents_device(None, 0, C.byref(p)) == L.FYX_ERR_INVALID_ARGUMENT
