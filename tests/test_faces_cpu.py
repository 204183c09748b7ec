"""Faces in the output arena (DCB_FACES_ARENA) without a GPU: the layout of the faces regions, the state and argument
checks, where each mesh's faces come from, and the host's location of plain sequential indices -- the ATTRIBUTES offset
and every framing status must be what the host decode gives."""
import ctypes as C
import os

import numpy as np
import pytest

import draco_sharp_b200 as D
import drc_writer as W
import faces_ref as F
from draco_sharp_b200 import _native as N
from oracle import pyoracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ERR_MAPS, ERR_STATE, ERR_ARG = -14, -104, -100


def _house():
    return np.fromfile(os.path.join(GOLD, "house_04.obj.drc"), dtype=np.uint8)


def _mixed():
    """point cloud, the house (Edgebreaker), sequential meshes of every index coding"""
    bufs = [np.frombuffer(W.point_cloud(50, F.attrs(50, 1)), dtype=np.uint8), _house()]
    bufs.append(F.mesh(F.grid_faces(7, 6), 42, 0, "raw", seed=2))
    bufs.append(F.mesh(F.grid_faces(7, 6), 42, 0, "tagged", seed=3))
    bufs.append(F.mesh(F.grid_faces(9, 9), 81, 1, seed=4))
    bufs.append(F.mesh(F.grid_faces(20, 15), 300, 1, seed=5))
    bufs.append(F.mesh(F.strip_faces(70000, 40), 70000, 1, with_attrs=False))
    bufs.append(F.mesh(F.strip_faces((1 << 21) + 5, 200), (1 << 21) + 5, 1, with_attrs=False))
    bufs.append(F.mesh([], 30, 1, seed=6))
    return bufs


def _index(bufs, faces, order_points=False):
    bt = D.index_only(bufs)
    if order_points:
        bt.set_output_order(True)
    if faces:
        bt.set_face_output(True)
    for k in range(len(bufs)):
        if bt.buffer_info(k).needs_connectivity:
            bt.host_connectivity(k)
    bt.finish()
    return bt


@pytest.mark.parametrize("order_points", [False, True])
def test_faces_regions_extend_the_arena_and_keep_attribute_offsets(order_points):
    bufs = _mixed()
    off = _index(bufs, False, order_points)
    on = _index(bufs, True, order_points)
    regions = []
    attr_end = 0
    for k, b in enumerate(bufs):
        bi = on.buffer_info(k)
        assert bi.status == 0 and off.buffer_info(k).status == 0
        for a in range(bi.n_attrs):
            x, y = off.attr_info(k, a), on.attr_info(k, a)
            assert (x.out_off, x.out_bytes) == (y.out_off, y.out_bytes)
            attr_end = max(attr_end, y.out_off + y.out_bytes)
        fi = on.face_info(k)
        assert off.face_info(k).source == 0 and off.face_info(k).out_bytes == 0
        if bi.geometry_type == 0:
            assert (fi.source, fi.out_bytes, fi.n_faces) == (0, 0, 0)
            continue
        o = O.decode(b)
        assert fi.n_faces == o.faces.shape[0] and fi.out_bytes == 12 * fi.n_faces and fi.out_off % 128 == 0
        regions.append((fi.out_off, fi.out_bytes))
    regions.sort()
    assert regions[0][0] >= attr_end
    for (a, n), (b2, _) in zip(regions, regions[1:]):
        assert a + n <= b2
    assert on.out_bytes - off.out_bytes == sum((n + 127) // 128 * 128 for _, n in regions)
    off.free()
    on.free()


def test_sources():
    bufs = _mixed()
    bt = _index(bufs, True)
    # point cloud: none; Edgebreaker and Tagged index differences: host; Raw index differences and plain indices: GPU
    assert [bt.face_info(k).source for k in range(len(bufs))] == [0, 1, 2, 1, 2, 2, 2, 2, 2]
    for k in (2, 4, 5, 6, 7, 8):  # the GPU decodes them: not on the host
        n = C.c_uint64(0)
        assert N.lib().dcb_mesh_faces(bt.h, k, None, 0, C.byref(n)) == ERR_STATE
    assert np.array_equal(bt.faces(3), O.decode(bufs[3]).faces)
    bt.free()


def test_state_and_argument_checks():
    bufs = _mixed()
    bt = _index(bufs, True)
    assert N.lib().dcb_set_face_output(bt.h, 2) == ERR_ARG
    assert N.lib().dcb_set_face_output(None, 1) == ERR_ARG
    assert N.lib().dcb_get_face_info(bt.h, len(bufs), C.byref(N.FaceInfo())) == ERR_ARG
    outs = (C.c_void_p * 1)()
    assert N.lib().dcb_decode_scatter(None, bt.h, outs, 1, 0) == ERR_STATE  # no slot for faces
    # indices located for the GPU are not on the host: the mode cannot be turned off any more
    assert N.lib().dcb_set_face_output(bt.h, 0) == ERR_STATE
    bt.free()
    # without such buffers, turning the mode off re-lays out the arena without the regions
    bt = _index(bufs[:2] + bufs[3:4], True)
    with_faces = bt.out_bytes
    bt.set_face_output(False)
    assert bt.out_bytes < with_faces and all(bt.face_info(k).source == 0 for k in range(3))
    bt.free()


def test_meshes_without_faces_fail_with_maps():
    house = _house()
    probe = D.index_only([house])
    probe.host_connectivity(0)
    probe.finish()
    n_dec = probe.buffer_info(0).n_attr_decoders
    maps = [[probe.mesh_map(0, d, w).copy() for w in range(4)] for d in range(n_dec)]
    aoff, npts = probe.buffer_info(0).attr_section_off, probe.buffer_info(0).n_points
    probe.free()
    seq = F.mesh(F.grid_faces(5, 4), 20, 1)
    seq_off = O.decode(seq).attr_section_off
    for faces in ("none", "null", "explicit"):
        bt = D.index_only([house, seq])
        bt.set_face_output(True)
        bt.set_attr_section(0, aoff, npts)
        for d in range(n_dec):
            bt.set_mesh_maps(0, d, *maps[d])
        if faces == "null":
            bt.set_mesh_faces(0, None)
        elif faces == "explicit":
            bt.set_mesh_faces(0, maps[0][1].reshape(-1, 3))
        bt.set_attr_section(1, seq_off, 20)  # caller-installed sequential connectivity: no faces
        bt.finish()
        assert bt.status(0) == (ERR_MAPS if faces == "none" else 0)
        assert bt.status(1) == ERR_MAPS
        if faces != "none":
            fi = bt.face_info(0)
            assert (fi.source, fi.n_faces) == (1, maps[0][1].size // 3)
        if faces == "none":  # faces installed after dcb_index_finish: the buffer is indexed again
            bt.set_mesh_faces(0, None)
            assert bt.status(0) == 0 and bt.face_info(0).source == 1
        bt.free()


@pytest.mark.parametrize("method,n_points,n_faces", [(1, 20, 0), (1, 200, 30), (1, 300, 40), (1, 60000, 40), (1, 70000, 40),
                                                     (1, 70000, 3000), (1, (1 << 21) - 1, 200), (1, (1 << 21) + 5, 200),
                                                     (0, 300, 40), (0, 70000, 3000)])
def test_located_attribute_offset_equals_the_host_decode(method, n_points, n_faces):
    faces = F.strip_faces(n_points, n_faces) if n_faces else []
    b = F.mesh(faces, n_points, method, with_attrs=n_points < 1000)
    o = O.decode(b)
    assert o.status == 0
    off, on = _index([b], False), _index([b], True)
    for bt in (off, on):
        bi = bt.buffer_info(0)
        assert bi.status == 0 and bi.attr_section_off == o.attr_section_off and bi.n_points == n_points
    fi = on.face_info(0)
    assert (fi.source, fi.n_faces) == (2, n_faces)
    off.free()
    on.free()


def _status(b, faces):
    bt = D.index_only([b])
    if faces:
        bt.set_face_output(True)
    if bt.buffer_info(0).status == 0:
        bt.host_connectivity(0)
        bt.finish()
    s = bt.buffer_info(0).status
    bt.free()
    return s


def _framing_cases():
    cases = []
    for method, n_points, faces in ((0, 30, F.grid_faces(6, 5)), (1, 30, F.grid_faces(6, 5)), (1, 300, F.grid_faces(20, 15)),
                                    (1, 70000, F.strip_faces(70000, 40)), (1, (1 << 21) + 5, F.strip_faces((1 << 21) + 5, 200))):
        good = bytearray(W.sequential_mesh(faces, n_points, [], method, "raw"))
        method_at = 11 + len(W.varint(len(faces))) + len(W.varint(n_points))
        bad = bytearray(good); bad[method_at] = 7  # connectivity method 7 (:81)
        cases.append(bytes(bad))
        idx_end = len(good) - 2  # ATTRIBUTES of point_cloud(n, []): n_dec = 1, one decoder without attributes
        for cut in sorted({11, 12, method_at, method_at + 1, 20, 40, (method_at + idx_end) // 2, idx_end - 5, idx_end - 1}):
            if 0 < cut < len(good):
                cases.append(bytes(good[:cut]))
    # (a running index out of range is no framing error: with Raw differences located, the GPU finds it -- test_faces_gpu.py)
    # varint indices (65536 <= points < 2^21): a varint of 10 continuation bytes (too long), one of 10 bytes (the longest
    # there is), and both cut inside the run
    for run in (10, 9):
        body = b"DRACO" + bytes([2, 2, 1, 0, 0, 0]) + W.varint(1) + W.varint(70000) + bytes([1])
        body += W.varint(5) + bytes([0x80] * run) + (b"" if run == 10 else b"\x01") + W.varint(7)
        cases.append(body + W.point_cloud(70000, [])[15:])
        cases.append(body[:-3])
    return cases


def test_framing_statuses_equal_the_host_decode():
    failed = 0
    for c in _framing_cases():
        b = np.frombuffer(c, dtype=np.uint8)
        host, located = _status(b, False), _status(b, True)
        assert located == host, (len(c), host, located)
        failed += host < 0
    assert failed >= 40
