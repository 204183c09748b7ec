"""-m gpu: point order (DCB_ORDER_POINTS) end to end.  Every attribute of an Edgebreaker mesh must equal the NumPy
gather (tests/point_order_ref.py) of the oracle's entry-order output through the oracle's faces and maps; point clouds
and sequential meshes keep their entry-order bytes; malformed maps fail their own buffer."""
import ctypes as C
import hashlib
import os
import struct

import numpy as np
import pytest

import draco_sharp_b200 as D
import drc_writer as W
from draco_sharp_b200 import _native as N
from oracle import pyoracle as O
from point_order_ref import gather_rows, point_map

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ERR_MAPS, ERR_STATE = -14, -104
POS_SHA = "028840c055ebfbc5b9a3a04b28d2fc5d0f9cae9c12821f030a815a0826bdcb37"
UV_SHA = "26bd6cc9ae35d081caba5b2061dd9d6d049a66c9050f7c5b9cfdc345c3c8449a"


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _house():
    return np.fromfile(os.path.join(GOLD, "house_04.obj.drc"), dtype=np.uint8)


def _mesh_buffer(attr_section):
    head = b"DRACO" + bytes([2, 2, 1, 1]) + struct.pack("<H", 0) + bytes([2]) + b"\xAA" * 37  # connectivity: host business
    return np.frombuffer(head + attr_section, dtype=np.uint8), len(head)


def _expected(ref, faces, maps, n_points, decs):
    """Point-order bytes of every attribute of an oracle result."""
    out = []
    for a, d in zip(ref.attrs, decs):
        m = point_map(faces, maps[d]["corner_to_vertex"], maps[d]["vertex_to_data"], n_points)
        raw = a.out.view(np.uint8)
        out.append(gather_rows(raw, raw.size // max(a.n_entries, 1), m))
    return out


def _attr_bytes(batch, out, k):
    return [out[ai.out_off: ai.out_off + ai.out_bytes] for ai in (batch.attr_info(k, a) for a in range(batch.buffer_info(k).n_attrs))]


def _decode_caller_maps(dec, bufs, conn, points=True):
    """conn[k]: (attr_section_off, n_points, maps, faces) of mesh k, or None (point cloud / host helper)."""
    batch = dec.index(bufs)
    if points:
        batch.set_output_order(True)
    for k, c in enumerate(conn):
        if c is None:
            if batch.buffer_info(k).needs_connectivity:
                batch.host_connectivity(k)
            continue
        off, n_points, maps, f = c
        batch.set_attr_section(k, off, n_points)
        for d, m in enumerate(maps):
            batch.set_mesh_maps(k, d, m["opposite"], m["corner_to_vertex"], m["data_to_corner"], m["vertex_to_data"])
        batch.set_mesh_faces(k, f)
    batch.finish()
    out, _ = dec.decode(batch)
    return batch, out


def test_house_whole_in_point_order(gpu_decoder):
    b = _house()
    o = O.decode(b)
    (d,) = gpu_decoder.decode_batch([b], point_order=True)
    assert d.ok and d.points_count == 3220 and np.array_equal(d.faces, o.faces)
    bt = D.index_only([b])
    bt.host_connectivity(0)
    bt.finish()
    decs = [bt.attr_info(0, a).decoder_id for a in range(3)]
    bt.free()
    want = _expected(o, o.faces, o.maps, o.n_points, decs)
    for a, w in zip(d.attributes, want):
        assert a.point_ordered and a.values.shape[0] == 3220
        assert np.array_equal(a.buffer, w)
    tri = d.get_named_attribute(0).values[d.faces]
    assert tri.shape == (2588, 3, 3)
    # entry order in the same process: the SHA-256 goldens
    (e,) = gpu_decoder.decode_batch([b])
    assert sha(e.attributes[0].buffer) == POS_SHA and sha(e.attributes[1].buffer) == UV_SHA
    assert not e.attributes[0].point_ordered and e.attributes[0].values.shape == (1775, 3)
    # the caller's connectivity (the oracle's maps + faces) gives the same bytes as the host helper
    batch, out = _decode_caller_maps(gpu_decoder, [b], [(o.attr_section_off, o.n_points, o.maps, o.faces)])
    assert batch.status(0) == 0
    for got, a in zip(_attr_bytes(batch, out, 0), d.attributes):
        assert np.array_equal(got, a.buffer)
    batch.free()


def _section(kind, scheme, o, rng):
    """An ATTRIBUTES section over the house's connectivity (decoders 0 and 1 of the sample) for one predictor."""
    n0, n1 = o.maps[0]["data_to_corner"].size, o.maps[1]["data_to_corner"].size
    sec = bytearray([2, 0xFF, 0, 0, 0, 1, 0])
    if kind == "parallelogram":
        sec += W.varint(2) + bytes([0, 9, 3, 0]) + W.varint(0) + bytes([4, 2, 1, 0]) + W.varint(1) + bytes([2, 1])
        sec += W.varint(1) + bytes([3, 9, 2, 0]) + W.varint(2) + bytes([2])
        sec += W.portable_int(rng.integers(-30, 31, size=n0 * 3), 3, 1, 1, scheme, W.wrap_data(0, 4095), num_bytes=2)
        sec += W.portable_int(rng.integers(-3, 4, size=n0), 1, 1, 1, scheme, W.wrap_data(0, 255), num_bytes=1)
        sec += W.quant_params([1.0, 2.0, 3.0], 10.0, 12)
        sec += W.portable_int(rng.integers(-9, 10, size=n1 * 2), 2, 1, 1, scheme, W.wrap_data(0, 1023), num_bytes=2)
        sec += W.quant_params([0.0, 0.0], 1.0, 10)
    elif kind == "cmp":
        def cmp(values, nc, m, bits):
            corr, crease = W.cmp_encode(values, nc, m, 0, (1 << bits) - 1, rng, 0.3)
            return W.portable_int(corr, nc, 4, 1, scheme, W.cmp_data(crease, 0, (1 << bits) - 1), num_bytes=4)
        sec += W.varint(1) + bytes([0, 9, 3, 0]) + W.varint(0) + bytes([2])
        sec += W.varint(1) + bytes([3, 9, 2, 0]) + W.varint(1) + bytes([2])
        sec += cmp(rng.integers(0, 4096, size=n0 * 3), 3, o.maps[0], 12) + W.quant_params([1.0, 2.0, 3.0], 10.0, 12)
        sec += cmp(rng.integers(0, 1024, size=n1 * 2), 2, o.maps[1], 10) + W.quant_params([0.0, 0.0], 1.0, 10)
    elif kind == "texcoords":
        sec += W.varint(1) + bytes([0, 9, 3, 0]) + W.varint(0) + bytes([2])
        sec += W.varint(1) + bytes([3, 9, 2, 0]) + W.varint(1) + bytes([2])
        sec += W.portable_int(rng.integers(-30, 31, size=n0 * 3), 3, 1, 1, scheme, W.wrap_data(0, 4095), num_bytes=4)
        sec += W.quant_params([1.0, 2.0, 3.0], 10.0, 12)
        sec += W.portable_int(rng.integers(-9, 10, size=n1 * 2), 2, 5, 1, scheme, W.tex_coords_data(rng.integers(0, 2, size=3300), 0, 1023),
                              num_bytes=4)
        sec += W.quant_params([0.0, 0.0], 1.0, 10)
    elif kind == "geometric":
        from test_geometric_normal_cpu import normals_section
        return normals_section(rng.integers(-40, 41, size=n0 * 3), rng.integers(0, 1024, size=n1 * 2), rng.integers(0, 2, size=n1), 10,
                               12, 1, scheme)
    elif kind == "octahedral":
        sec += W.varint(1) + bytes([0, 9, 3, 0]) + W.varint(0) + bytes([2])
        sec += W.varint(1) + bytes([1, 9, 3, 0]) + W.varint(1) + bytes([3])
        sec += W.portable_int(rng.integers(-30, 31, size=n0 * 3), 3, 1, 1, scheme, W.wrap_data(0, 4095), num_bytes=4)
        sec += W.quant_params([1.0, 2.0, 3.0], 10.0, 12)
        sec += W.portable_int(rng.integers(-20, 21, size=n1 * 2), 2, 0, 3, scheme, struct.pack("<ii", 1023, 511), num_bytes=4)
        sec += bytes([10])
    elif kind == "generic7":  # difference-coded integer attribute with seven components
        sec += W.varint(1) + bytes([0, 9, 3, 0]) + W.varint(0) + bytes([2])
        sec += W.varint(1) + bytes([4, 4, 7, 0]) + W.varint(1) + bytes([1])
        sec += W.portable_int(rng.integers(-30, 31, size=n0 * 3), 3, 1, 1, scheme, W.wrap_data(0, 4095), num_bytes=4)
        sec += W.quant_params([1.0, 2.0, 3.0], 10.0, 12)
        sec += W.portable_int(rng.integers(-50, 51, size=n1 * 7), 7, 0, 1, scheme, W.wrap_data(0, 60000), num_bytes=4)
    return bytes(sec)


KINDS = ["parallelogram", "cmp", "texcoords", "geometric", "octahedral", "generic7"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("scheme", ["raw", "tagged", "uncompressed"])
def test_every_predictor_over_the_house_connectivity(gpu_decoder, kind, scheme):
    b = _house()
    o = O.decode(b)
    rng = np.random.default_rng(KINDS.index(kind) * 3 + len(scheme))
    buf, aoff = _mesh_buffer(_section(kind, scheme, o, rng))
    maps = [o.maps[0], o.maps[1]]
    ref = O.decode(buf, maps, aoff, o.n_points)
    assert ref.status == 0
    batch, out = _decode_caller_maps(gpu_decoder, [buf], [(aoff, o.n_points, maps, o.faces)])
    assert batch.status(0) == 0
    decs = [batch.attr_info(0, a).decoder_id for a in range(len(ref.attrs))]
    for a, (got, want) in enumerate(zip(_attr_bytes(batch, out, 0), _expected(ref, o.faces, maps, o.n_points, decs))):
        assert np.array_equal(got, want), (kind, scheme, a)
    batch.free()


@pytest.mark.parametrize("w,h", [(2, 2), (17, 9), (300, 300), (1000, 1000)])
def test_grid_meshes_faces_omitted_equal_explicit_faces(gpu_decoder, w, h):
    from draco_sharp_b200 import synth_gen as G
    topo = G.grid_topology(w, h)
    meshes = [G.grid_mesh(w, h, topo, seed=300 + k, scheme=k % 2 - 1) for k in range(3)]
    bufs = [m[0] for m in meshes]
    faces = np.asarray(topo["corner_to_vertex"], dtype=np.uint32)
    res = []
    for f in (None, faces):
        batch, out = _decode_caller_maps(gpu_decoder, bufs, [(m[1], w * h, [topo], f) for m in meshes])
        res.append([_attr_bytes(batch, out, k)[0].copy() for k in range(len(bufs))])
        ent = [O.decode(m[0], [topo], m[1], w * h) for m in meshes]
        for k in range(len(bufs)):
            assert batch.status(k) == 0
            rows = ent[k].attrs[0].out.view(np.uint8).reshape(-1, 12)
            assert np.array_equal(res[-1][k], rows[np.asarray(topo["vertex_to_data"])].ravel())
        batch.free()
    for x, y in zip(*res):
        assert np.array_equal(x, y)


def _seq_and_cloud():
    rng = np.random.default_rng(8)
    w, h = 40, 30
    n = w * h
    faces = [(y * w + x, y * w + x + 1, (y + 1) * w + x) for y in range(h - 1) for x in range(w - 1)]
    attrs = [dict(att_type=0, data_type=9, nc=3, seq_type=2,
                  portable=W.portable_int(rng.integers(-20, 21, size=n * 3), 3, 0, 1, "tagged", W.wrap_data(0, 4095), num_bytes=2),
                  xform=W.quant_params([0.0, 1.0, 2.0], 8.0, 12)),
             dict(att_type=2, data_type=2, nc=3, seq_type=1,
                  portable=W.portable_int(rng.integers(-3, 4, size=n * 3), 3, 0, 1, "raw", W.wrap_data(0, 255)))]
    seq = np.frombuffer(W.sequential_mesh(faces, n, attrs, 0, "raw"), dtype=np.uint8)
    cloud = np.frombuffer(W.point_cloud(n, attrs), dtype=np.uint8)
    return seq, cloud


@pytest.mark.parametrize("bad", ["point", "vertex", "entry"])
def test_mixed_batch_and_malformed_maps(gpu_decoder, bad):
    b = _house()
    o = O.decode(b)
    seq, cloud = _seq_and_cloud()
    maps = [dict(m) for m in o.maps]
    faces = o.faces.copy()
    if bad == "point":
        faces[100, 1] = o.n_points
    elif bad == "vertex":
        maps[1] = dict(maps[1], corner_to_vertex=maps[1]["corner_to_vertex"].copy())
        maps[1]["corner_to_vertex"][7] = maps[1]["vertex_to_data"].size
    else:
        maps[0] = dict(maps[0], vertex_to_data=maps[0]["vertex_to_data"].copy())
        maps[0]["vertex_to_data"][o.maps[0]["corner_to_vertex"][5]] = o.maps[0]["data_to_corner"].size
    bufs = [cloud, seq, b, b, b, cloud]
    conn = [None, None, None, (o.attr_section_off, o.n_points, maps, faces), None, None]
    pts, out_p = _decode_caller_maps(gpu_decoder, bufs, conn)
    ent, out_e = _decode_caller_maps(gpu_decoder, bufs, [None] * 3 + [(o.attr_section_off, o.n_points, o.maps, o.faces)] + [None] * 2,
                                     points=False)
    assert [pts.status(k) for k in range(6)] == [0, 0, 0, ERR_MAPS, 0, 0]
    for k in (0, 1, 5):  # clouds and sequential meshes: entry-order bytes
        for x, y in zip(_attr_bytes(pts, out_p, k), _attr_bytes(ent, out_e, k)):
            assert np.array_equal(x, y), k
    decs = [pts.attr_info(2, a).decoder_id for a in range(3)]
    want = _expected(o, o.faces, o.maps, o.n_points, decs)
    for k in (2, 4):
        for x, y in zip(_attr_bytes(pts, out_p, k), want):
            assert np.array_equal(x, y), k
    pts.free()
    ent.free()


def test_conflicting_corners_take_the_highest_corner(gpu_decoder):
    """Caller faces that merge two points whose corners carry different entries: the higher corner index wins."""
    b = _house()
    o = O.decode(b)
    faces = o.faces.copy().ravel()
    a, z = int(faces[10]), int(faces[4000])
    faces[faces == z] = a               # point z's corners now say point a: z is unreferenced
    batch, out = _decode_caller_maps(gpu_decoder, [b], [(o.attr_section_off, o.n_points, o.maps, faces)])
    assert batch.status(0) == 0
    decs = [batch.attr_info(0, k).decoder_id for k in range(3)]
    want = _expected(o, faces, o.maps, o.n_points, decs)
    got = _attr_bytes(batch, out, 0)
    for x, y in zip(got, want):
        assert np.array_equal(x, y)
    pos = got[0].reshape(-1, 12)
    assert not pos[z].any()             # unreferenced: zero row
    last = int(np.nonzero(faces == a)[0].max())
    e = o.maps[0]["vertex_to_data"][o.maps[0]["corner_to_vertex"][last]]
    assert np.array_equal(pos[a], o.attrs[0].out.view(np.uint8).reshape(-1, 12)[e])
    batch.free()


def _indexed_points(dec, bufs):
    batch = dec.index(bufs)
    batch.set_output_order(True)
    for k in range(len(bufs)):
        if batch.buffer_info(k).needs_connectivity:
            batch.host_connectivity(k)
    batch.finish()
    return batch


def test_delivery_paths(gpu_decoder):
    import torch
    b = _house()
    seq, cloud = _seq_and_cloud()
    bufs = [cloud, b, seq, b]
    ref, out = _decode_caller_maps(gpu_decoder, bufs, [None] * 4)
    assert [ref.status(k) for k in range(4)] == [0, 0, 0, 0]
    want = [x.copy() for k in range(4) for x in _attr_bytes(ref, out, k)]
    # decode_scatter: one caller array per attribute, sized by out_bytes
    infos = [ref.attr_info(k, a) for k in range(4) for a in range(ref.buffer_info(k).n_attrs)]
    outs = [np.zeros(ai.out_bytes, dtype=np.uint8) for ai in infos]
    batch = _indexed_points(gpu_decoder, bufs)
    ptrs = (C.c_void_p * len(outs))(*[x.ctypes.data for x in outs])
    N.check(N.lib().dcb_decode_scatter(gpu_decoder.ctx, batch.h, ptrs, len(outs), 0))
    for x, y in zip(outs, want):
        assert np.array_equal(x, y)
    batch.free()
    # upload + resident into a torch tensor of exactly out_bytes, twice, then download
    batch = _indexed_points(gpu_decoder, bufs)
    gpu_decoder.upload(batch)
    assert N.lib().dcb_set_output_order(batch.h, 0) == ERR_STATE
    t = torch.empty(batch.out_bytes, dtype=torch.uint8, device="cuda")
    got = []
    for _ in range(2):
        t.fill_(0xCD)
        gpu_decoder.decode_resident(batch, dev_out=t.data_ptr())
        got.append(t.cpu().numpy().copy())
    assert np.array_equal(got[0], got[1])
    host = np.zeros(batch.out_bytes, dtype=np.uint8)
    gpu_decoder.download(batch, host)
    assert np.array_equal(host, got[0])
    for ai, y in zip(infos, want):
        assert np.array_equal(host[ai.out_off: ai.out_off + ai.out_bytes], y)
    batch.free()
    # pipeline slices
    dec = D.DracoBatchDecoder([0, 0, 0])
    try:
        many = dec.decode_batch(bufs * 3, point_order=True)
    finally:
        dec.close()
    flat = [a.buffer for d in many for a in d.attributes]
    for k, x in enumerate(flat):
        assert np.array_equal(x, want[k % len(want)]), k


def test_distinct_devices(gpu_decoder):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    b = _house()
    seq, cloud = _seq_and_cloud()
    bufs = [cloud, b, seq, b] * 4
    one = gpu_decoder.decode_batch(bufs, point_order=True)
    dec = D.DracoBatchDecoder([0, 1])
    try:
        two = dec.decode_batch(bufs, point_order=True)
    finally:
        dec.close()
    for x, y in zip(one, two):
        assert x.ok and y.ok
        for a, c in zip(x.attributes, y.attributes):
            assert np.array_equal(a.buffer, c.buffer)
