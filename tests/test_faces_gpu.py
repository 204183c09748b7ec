"""-m gpu: faces in the output arena (DCB_FACES_ARENA) end to end.  The faces region of every mesh must equal the oracle's
faces; attributes must be byte-identical to the same batch decoded with the mode off, in both output orders; every
delivery path must give the same arena."""
import ctypes as C
import os

import numpy as np
import pytest

import draco_sharp_b200 as D
import drc_writer as W
import faces_ref as F
from draco_sharp_b200 import _native as N
from oracle import pyoracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ERR_STATE = -104


def _house():
    return np.fromfile(os.path.join(GOLD, "house_04.obj.drc"), dtype=np.uint8)


def _decode(dec, bufs, faces, points=False, conn=None):
    """conn[k]: (attr_section_off, n_points, maps, faces or None for the NULL form) of a caller-decoded Edgebreaker mesh"""
    batch = dec.index(bufs)
    if points:
        batch.set_output_order(True)
    if faces:
        batch.set_face_output(True)
    for k in range(len(bufs)):
        c = conn[k] if conn else None
        if c is not None:
            off, n_points, maps, f = c
            batch.set_attr_section(k, off, n_points)
            for d, m in enumerate(maps):
                batch.set_mesh_maps(k, d, *m)
            batch.set_mesh_faces(k, f)
        elif batch.buffer_info(k).needs_connectivity:
            batch.host_connectivity(k)
    batch.finish()
    out, _ = dec.decode(batch)
    return batch, out


def _faces(batch, out, k):
    fi = batch.face_info(k)
    return out[fi.out_off: fi.out_off + fi.out_bytes].view(np.uint32).reshape(-1, 3)


def _attrs(batch, out, k):
    return [out[ai.out_off: ai.out_off + ai.out_bytes].copy()
            for ai in (batch.attr_info(k, a) for a in range(batch.buffer_info(k).n_attrs))]


def _sequential_cases():
    """(buffer, expected source): every index coding, point counts on both sides of 256, 65536 and 2^21, 0 faces, and
    varint runs of many 4 KiB chunks"""
    cases = [(F.mesh(F.grid_faces(6, 5), 30, 0, "raw", seed=1), 2), (F.mesh(F.grid_faces(6, 5), 30, 0, "tagged", seed=2), 1),
             (F.mesh(F.grid_faces(40, 30), 1200, 0, "raw", seed=3), 2), (F.mesh(F.grid_faces(40, 30), 1200, 0, "tagged", seed=4), 1),
             (F.mesh([], 30, 0, seed=5), 1), (F.mesh([], 30, 1, seed=6), 2)]
    for n in (255, 256, 65535, 65536, (1 << 21) - 1, 1 << 21):
        cases.append((F.mesh(F.strip_faces(n, min(301, n - 3)), n, 1, with_attrs=n < 1000, seed=n & 255), 2))
    cases.append((F.mesh(F.grid_faces(16, 16), 256, 1, seed=7), 2))
    cases.append((F.mesh(F.grid_faces(270, 250), 67500, 1, with_attrs=False), 2))  # ~400k varints: ~300 chunks
    cases.append((F.mesh(F.grid_faces(120, 100), 12000, 0, "raw", with_attrs=False), 2))  # ~71k symbols: 18 scan chunks
    return cases


def test_sequential_faces_equal_the_oracle(gpu_decoder):
    cases = _sequential_cases()
    bufs = [b for b, _ in cases]
    batch, out = _decode(gpu_decoder, bufs, True)
    for k, (b, src) in enumerate(cases):
        o = O.decode(b)
        assert o.status == 0 and batch.status(k) == 0, (k, o.status, batch.status(k))
        fi = batch.face_info(k)
        assert fi.source == src and fi.n_faces == o.faces.shape[0], k
        assert np.array_equal(_faces(batch, out, k), o.faces.reshape(-1, 3)), k
        for a, oa in enumerate(o.attrs):
            ai = batch.attr_info(k, a)
            assert np.array_equal(out[ai.out_off: ai.out_off + ai.out_bytes], oa.out.view(np.uint8).reshape(-1)), (k, a)
    batch.free()


def test_index_errors_fail_their_buffer_only(gpu_decoder):
    good = F.mesh(F.grid_faces(6, 5), 30, 1, seed=1)
    # Raw index differences that drop below zero (in the second scan chunk) and that pass INT32_MAX (steps of 2^18),
    # decoded and checked on the GPU; a Raw index payload and plain indices cut short (framing: the host)
    head = b"DRACO" + bytes([2, 2, 1, 0, 0, 0])
    tail = W.point_cloud(3, F.attrs(3, 1))[15:]
    syms = [0] * 5000 + [3] + [0] * 4
    neg = head + W.varint(len(syms) // 3) + W.varint(3) + bytes([0]) + W.symbols_raw(syms) + tail
    syms = [1 << 19] * 8193 + [0, 0]
    big = head + W.varint(len(syms) // 3) + W.varint(3) + bytes([0]) + W.symbols_raw(syms) + tail
    raw = W.sequential_mesh(F.grid_faces(20, 15), 300, [], 0)
    plain = W.sequential_mesh(F.strip_faces(70000, 300), 70000, [], 1)
    bad = (neg, big, raw[:len(raw) // 2], plain[:len(plain) - 40])
    bufs = [good] + [np.frombuffer(x, dtype=np.uint8) for x in bad] + [good]
    host = D.index_only(bufs)
    for k in range(len(bufs)):
        host.host_connectivity(k)
    batch, out = _decode(gpu_decoder, bufs, True)
    for k in range(1, len(bufs) - 1):
        assert batch.status(k) < 0 and batch.status(k) == host.buffer_info(k).status, k
        assert batch.face_info(k).source == 0
    for k in (0, len(bufs) - 1):
        assert batch.status(k) == 0 and np.array_equal(_faces(batch, out, k), O.decode(bufs[k]).faces.reshape(-1, 3))
    host.free()
    batch.free()


def _mixed():
    house = _house()
    probe = D.index_only([house])
    probe.host_connectivity(0)
    probe.finish()
    n_dec = probe.buffer_info(0).n_attr_decoders
    maps = [[probe.mesh_map(0, d, w).copy() for w in range(4)] for d in range(n_dec)]
    host_faces = probe.faces(0)
    conn_info = (probe.buffer_info(0).attr_section_off, probe.buffer_info(0).n_points)
    probe.free()
    bufs = [np.frombuffer(W.point_cloud(500, F.attrs(500, 9)), dtype=np.uint8), house, house, house]
    conn = [None, None, conn_info + (maps, host_faces), conn_info + (maps, None)]
    want = [None, host_faces, host_faces, maps[0][1].reshape(-1, 3)]
    for b, _ in _sequential_cases()[:8]:
        bufs.append(b)
        conn.append(None)
        want.append(O.decode(b).faces.reshape(-1, 3))
    return bufs, conn, want


@pytest.mark.parametrize("points", [False, True])
def test_mixed_batch_attributes_are_unchanged(gpu_decoder, points):
    bufs, conn, want = _mixed()
    b0, o0 = _decode(gpu_decoder, bufs, False, points, conn)
    b1, o1 = _decode(gpu_decoder, bufs, True, points, conn)
    for k in range(len(bufs)):
        assert b0.status(k) == 0 and b1.status(k) == 0, k
        x, y = _attrs(b0, o0, k), _attrs(b1, o1, k)
        assert len(x) == len(y) and all(np.array_equal(p, q) for p, q in zip(x, y)), k
        if want[k] is None:
            assert b1.face_info(k).source == 0
        else:
            assert np.array_equal(_faces(b1, o1, k), want[k]), k
    b0.free()
    b1.free()


def test_decode_batch_faces_in_arena(gpu_decoder):
    bufs, _, _ = _mixed()
    for points in (False, True):
        ref = gpu_decoder.decode_batch(bufs, point_order=points)
        got = gpu_decoder.decode_batch(bufs, point_order=points, faces_in_arena=True)
        for r, g in zip(ref, got):
            assert r.status == g.status == 0
            assert (r.faces is None) == (g.faces is None)
            if r.faces is not None:
                assert g.faces.dtype == np.uint32 and np.array_equal(r.faces, g.faces)


def _same_outputs(b0, o0, b1, o1, n):
    for k in range(n):
        assert b1.status(k) == 0, k
        assert np.array_equal(_faces(b0, o0, k), _faces(b1, o1, k)), k
        assert all(np.array_equal(x, y) for x, y in zip(_attrs(b0, o0, k), _attrs(b1, o1, k))), k


def test_delivery_paths(gpu_decoder):
    import torch
    bufs, conn, _ = _mixed()
    ref_batch, ref = _decode(gpu_decoder, bufs, True, True, conn)
    n = ref_batch.out_bytes
    # upload + resident into a caller's device buffer, twice, then download
    batch = gpu_decoder.index(bufs)
    batch.set_output_order(True)
    batch.set_face_output(True)
    for k, c in enumerate(conn):
        if c is None:
            if batch.buffer_info(k).needs_connectivity:
                batch.host_connectivity(k)
            continue
        batch.set_attr_section(k, c[0], c[1])
        for d, m in enumerate(c[2]):
            batch.set_mesh_maps(k, d, *m)
        batch.set_mesh_faces(k, c[3])
    batch.finish()
    gpu_decoder.upload(batch)
    assert N.lib().dcb_set_face_output(batch.h, N.DCB_FACES_NONE) == ERR_STATE  # the arena is laid out
    outs = (C.c_void_p * 1)()
    assert N.lib().dcb_decode_scatter(gpu_decoder.ctx, batch.h, outs, 1, 0) == ERR_STATE
    t = torch.empty(n, dtype=torch.uint8, device="cuda")
    for _ in range(2):
        t.fill_(0xEE)
        gpu_decoder.decode_resident(batch, dev_out=t.data_ptr())
        _same_outputs(ref_batch, ref, batch, t.cpu().numpy(), len(bufs))
    host = np.zeros(n, dtype=np.uint8)
    gpu_decoder.decode_resident(batch)
    gpu_decoder.download(batch, host)
    _same_outputs(ref_batch, ref, batch, host, len(bufs))
    batch.free()
    # pipeline slices: one device listed three times
    dec = D.DracoBatchDecoder([0, 0, 0])
    try:
        b3, o3 = _decode(dec, bufs, True, True, conn)
        _same_outputs(ref_batch, ref, b3, o3, len(bufs))
        b3.free()
    finally:
        dec.close()
    ref_batch.free()


def test_distinct_devices(gpu_decoder):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    bufs, conn, _ = _mixed()
    ref_batch, ref = _decode(gpu_decoder, bufs, True, True, conn)
    dec = D.DracoBatchDecoder([0, 1])
    try:
        b2, o2 = _decode(dec, bufs, True, True, conn)
        _same_outputs(ref_batch, ref, b2, o2, len(bufs))
        b2.free()
    finally:
        dec.close()
    ref_batch.free()
