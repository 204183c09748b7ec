"""Point order (DCB_ORDER_POINTS) without a device: the rule restated in NumPy from the oracle's faces and maps, checked
against invariants that do not come from the library, and the output layout, argument and state checks of the C ABI
(dcb_set_output_order, dcb_set_mesh_faces) on indexed batches."""
import os

import numpy as np
import pytest

import draco_sharp_b200 as D
import drc_writer as W
from draco_sharp_b200 import _native as N
from oracle import pyoracle as O
from point_order_ref import gather_rows, point_map, row_bytes

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ERR_ARG, ERR_STATE, ERR_MAPS = -100, -104, -14


def _house():
    return np.fromfile(os.path.join(GOLD, "house_04.obj.drc"), dtype=np.uint8)


def _half_step(a):
    return float(a.qrange) / ((1 << a.qbits) - 1) / 2


def test_reference_rule_on_the_house_sample():
    b = _house()
    o = O.decode(b)
    assert o.status == 0 and o.n_points == 3220
    bt = D.index_only([b])
    bt.host_connectivity(0)
    bt.finish()
    decs = [bt.attr_info(0, a).decoder_id for a in range(3)]
    bt.free()
    faces = o.faces.ravel()
    maps = [point_map(faces, m["corner_to_vertex"], m["vertex_to_data"], o.n_points) for m in o.maps]
    per_corner = [np.asarray(m["vertex_to_data"], np.int64)[np.asarray(m["corner_to_vertex"], np.int64)] for m in o.maps]
    # every corner's point maps to its vertex's entry (no conflicts in a well-formed mesh)
    for m, pc in zip(maps, per_corner):
        assert np.array_equal(m[faces], pc)
        assert (m >= 0).all()
    # the points are exactly the distinct tuples of per-decoder entries over the corners
    tuples = np.stack(per_corner, axis=1)
    assert np.unique(tuples, axis=0).shape[0] == o.n_points
    assert np.unique(np.stack(maps, axis=1), axis=0).shape[0] == o.n_points
    assert {tuple(t) for t in tuples} == {tuple(t) for t in np.stack(maps, axis=1)}
    # per-point positions / UVs lie within half a quantisation step of a line of the source OBJ
    for k, golden in ((0, "house_04_obj_vertices.npy"), (1, "house_04_obj_texcoords.npy")):
        a = o.attrs[k]
        vals = a.out.view(np.float32).reshape(a.n_entries, -1)[maps[decs[k]]].astype(np.float64)
        assert vals.shape == (3220, a.nc)
        ref = np.load(os.path.join(GOLD, golden)).astype(np.float64)
        dist = np.abs(vals[:, None, :] - ref[None, :, :]).max(axis=2).min(axis=1)
        assert dist.max() < _half_step(a), k


def test_reference_conflict_rule_and_unreferenced_points():
    faces = np.array([0, 1, 2, 0, 2, 3], dtype=np.uint32)        # point 0 on corners 0 and 3, point 4 on none
    c2v = np.array([0, 1, 2, 3, 2, 1], dtype=np.uint32)
    v2d = np.array([5, 6, 7, 8], dtype=np.int32)
    m = point_map(faces, c2v, v2d, 5)
    assert m.tolist() == [8, 6, 7, 6, -1]
    rows = gather_rows(np.arange(9 * 2, dtype=np.uint8), 2, m)
    assert rows.reshape(5, 2)[4].tolist() == [0, 0] and rows.reshape(5, 2)[0].tolist() == [16, 17]


def _infos(bt, k):
    return [bt.attr_info(k, a) for a in range(bt.buffer_info(k).n_attrs)]


def _fields(ai, skip=()):
    return tuple(getattr(ai, f) if f != "q_min" else tuple(ai.q_min) for f, _ in N.AttrInfo._fields_ if f not in skip)


def _seq_and_cloud():
    rng = np.random.default_rng(3)
    w, h = 12, 9
    n = w * h
    faces = [(y * w + x, y * w + x + 1, (y + 1) * w + x) for y in range(h - 1) for x in range(w - 1)]
    attrs = [dict(att_type=0, data_type=9, nc=3, seq_type=2,
                  portable=W.portable_int(rng.integers(-20, 21, size=n * 3), 3, 0, 1, "raw", W.wrap_data(0, 4095), num_bytes=2),
                  xform=W.quant_params([0.0, 1.0, 2.0], 8.0, 12)),
             dict(att_type=2, data_type=2, nc=3, seq_type=1,
                  portable=W.portable_int(rng.integers(-3, 4, size=n * 3), 3, 0, 1, "raw", W.wrap_data(0, 255)))]
    seq = np.frombuffer(W.sequential_mesh(faces, n, attrs, 0, "raw"), dtype=np.uint8)
    cloud = np.frombuffer(W.point_cloud(n, attrs), dtype=np.uint8)
    return seq, cloud


def _indexed(bufs, points, order_first=True):
    bt = D.index_only(bufs)
    if points and order_first:
        bt.set_output_order(True)
    for k in range(len(bufs)):
        if bt.buffer_info(k).needs_connectivity:
            bt.host_connectivity(k)
    bt.finish()
    if points and not order_first:
        bt.set_output_order(True)
    return bt


@pytest.mark.parametrize("order_first", [True, False])
def test_point_layout_of_the_house_next_to_clouds_and_sequential_meshes(order_first):
    seq, cloud = _seq_and_cloud()
    bufs = [cloud, seq, _house(), cloud, seq]
    ent = _indexed(bufs, False)
    pts = _indexed(bufs, True, order_first)
    for k in range(len(bufs)):
        assert pts.status(k) == ent.status(k) == 0
    # the house: 3,220 rows of every attribute
    for ai in _infos(pts, 2):
        assert ai.out_bytes == 3220 * row_bytes(ai) and ai.out_off % 128 == 0
    assert [ai.n_entries for ai in _infos(pts, 2)] == [1775, 3220, 1775]
    # in front of the house: identical info; behind it: identical but for the offset
    for k in (0, 1):
        assert [_fields(a) for a in _infos(pts, k)] == [_fields(a) for a in _infos(ent, k)]
    for k in (3, 4):
        assert [_fields(a, ("out_off",)) for a in _infos(pts, k)] == [_fields(a, ("out_off",)) for a in _infos(ent, k)]
    spans = sorted((ai.out_off, ai.out_off + ai.out_bytes) for k in range(len(bufs)) for ai in _infos(pts, k))
    for (a0, a1), (b0, _) in zip(spans, spans[1:]):
        assert a1 <= b0
    assert pts.out_bytes == (spans[-1][1] + 127) // 128 * 128
    assert pts.out_bytes > ent.out_bytes
    # back to entry order: the entry layout again
    pts.set_output_order(False)
    assert pts.out_bytes == ent.out_bytes
    for k in range(len(bufs)):
        assert [_fields(a) for a in _infos(pts, k)] == [_fields(a) for a in _infos(ent, k)]
    ent.free()
    pts.free()


def test_arguments_and_state():
    seq, cloud = _seq_and_cloud()
    bt = D.index_only([cloud, _house(), seq])
    lib = N.lib()
    assert lib.dcb_set_output_order(bt.h, 2) == ERR_ARG
    assert lib.dcb_set_output_order(bt.h, -1) == ERR_ARG
    assert lib.dcb_set_output_order(None, 1) == ERR_ARG
    assert lib.dcb_set_mesh_faces(bt.h, 0, None, 0) == ERR_STATE      # point cloud
    assert lib.dcb_set_mesh_faces(bt.h, 2, None, 0) == ERR_STATE      # sequential mesh
    assert lib.dcb_set_mesh_faces(bt.h, 1, None, 3) == ERR_ARG        # NULL faces with a count
    assert lib.dcb_set_mesh_faces(bt.h, 7, None, 0) == ERR_ARG
    assert lib.dcb_set_mesh_faces(bt.h, 1, None, 0) == 0              # the NULL form
    bt.free()


def test_face_checks_fail_one_buffer_only():
    b = _house()
    o = O.decode(b)
    bt = D.index_only([b, b, b, b])
    bt.set_output_order(True)
    for k in range(4):
        bt.set_attr_section(k, o.attr_section_off, o.n_points)
        for d, m in enumerate(o.maps):
            bt.set_mesh_maps(k, d, m["opposite"], m["corner_to_vertex"], m["data_to_corner"], m["vertex_to_data"])
    bt.set_mesh_faces(0, o.faces)
    bt.set_mesh_faces(1, o.faces[:-1])          # one face short of n_corners
    # buffer 2: no faces at all
    bt.set_mesh_faces(3, None)                  # the NULL form: 3 * n_faces = n_corners of every decoder
    bt.finish()
    assert [bt.status(k) for k in range(4)] == [0, ERR_MAPS, ERR_MAPS, 0]
    assert bt.attr_info(0, 0).out_bytes == 3220 * 12
    # fixing the faces re-runs the check; entry order needs no faces
    bt.set_mesh_faces(1, o.faces)
    assert [bt.status(k) for k in range(4)] == [0, 0, ERR_MAPS, 0]
    bt.set_output_order(False)
    assert [bt.status(k) for k in range(4)] == [0, 0, 0, 0]
    assert bt.attr_info(0, 0).out_bytes == 1775 * 12
    bt.free()
