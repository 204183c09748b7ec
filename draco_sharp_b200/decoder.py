"""Host-side mirror of the reference's decoder interface for the GPU batch path.

The reference exposes `DracoDecoder.Decode(path | byte[] | BinaryReader) -> Draco`
(src/Draco/IO/DracoDecoder.cs:8,14,19; result type src/Draco/Draco.cs:9-15 with Header,
Attributes / ConnectedData holding `PointAttribute`s whose `Buffer` is a `DataBuffer` byte array,
src/Draco/IO/Attributes/GeometryAttribute.cs:10-17, PointAttribute.cs:7-63).  The C# drop-in
(csharp/DracoBatchDecoder.cs) keeps those types and adds `DecodeBatch`; this module is the same
thing for Python callers, used by the tests and by bench.py.  It calls the C ABI only
(include/dracob200.h): there is no CPU decode path, and construction fails with
DCB_ERR_NO_DEVICE when no B200 is present.
"""
import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _native as N

# DataType enum -> numpy dtype (src/Draco/IO/Enums/DataType.cs)
NP_DTYPES = {1: np.int8, 2: np.uint8, 3: np.int16, 4: np.uint16, 5: np.int32, 6: np.uint32, 7: np.int64,
             8: np.uint64, 9: np.float32, 10: np.float64, 11: np.uint8}
GEOMETRY_ATTRIBUTE_TYPES = {0: "Position", 1: "Normal", 2: "Color", 3: "TexCoord", 4: "Generic"}


@dataclass
class DracoHeader:  # src/Draco/DracoHeader.cs:5-23
    major_version: int
    minor_version: int
    encoder_type: int    # 0 point cloud, 1 triangular mesh
    encoder_method: int  # 0 sequential, 1 Edgebreaker
    flags: int


@dataclass
class PointAttribute:  # src/Draco/IO/Attributes/PointAttribute.cs + GeometryAttribute.cs
    attribute_type: int
    data_type: int
    num_components: int
    normalized: bool
    unique_id: int
    byte_stride: int
    unique_entries_count: int
    buffer: np.ndarray            # uint8 view of the attribute bytes (DataBuffer)
    info: N.AttrInfo = None
    point_ordered: bool = False   # rows are points (DCB_ORDER_POINTS on an Edgebreaker mesh), not unique entries

    @property
    def rows(self):
        return self.buffer.size // self.byte_stride if self.byte_stride else 0

    @property
    def values(self):
        """(rows, num_components): unique entries in entry order, or one row per point when point_ordered."""
        dt = NP_DTYPES[self.data_type]
        return self.buffer.view(dt).reshape(self.rows, self.num_components)


@dataclass
class Draco:  # src/Draco/Draco.cs:9-15
    header: Optional[DracoHeader]
    status: int
    points_count: int = 0
    attributes: List[PointAttribute] = field(default_factory=list)
    faces: Optional[np.ndarray] = None  # meshes: (n_faces, 3) point ids, Mesh.cs:5-19

    @property
    def ok(self):
        return self.status == 0

    def get_named_attribute(self, att_type):  # PointCloud.cs:19-58
        for a in self.attributes:
            if a.attribute_type == att_type:
                return a
        return None


class Batch:
    """An indexed batch (dcb_batch): stream descriptors on the host, arenas on the device."""

    def __init__(self, dec, handle, n_bufs, keep):
        self._dec = dec
        self.h = handle
        self.n_bufs = n_bufs
        self._keep = keep  # input buffers must outlive upload
        self.point_order = False
        self.faces_in_arena = False

    def free(self):
        if self.h:
            N.lib().dcb_batch_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    @property
    def out_bytes(self):
        return int(N.lib().dcb_batch_out_bytes(self.h))

    @property
    def dbg_bytes(self):
        return int(N.lib().dcb_batch_dbg_bytes(self.h))

    @property
    def in_bytes(self):
        return int(N.lib().dcb_batch_in_bytes(self.h))

    @property
    def points(self):
        return int(N.lib().dcb_batch_points(self.h))

    @property
    def algo_bytes(self):
        return int(N.lib().dcb_batch_algo_bytes(self.h))

    def buffer_info(self, k):
        bi = N.BufferInfo()
        N.check(N.lib().dcb_get_buffer_info(self.h, k, C.byref(bi)))
        return bi

    def attr_info(self, k, a):
        ai = N.AttrInfo()
        N.check(N.lib().dcb_get_attr_info(self.h, k, a, C.byref(ai)))
        return ai

    def status(self, k):
        return int(N.lib().dcb_status(self.h, k))

    def set_attr_section(self, k, off, n_points):
        N.check(N.lib().dcb_set_attr_section(self.h, k, off, n_points))

    def set_mesh_maps(self, k, dec, opposite, corner_to_vertex, data_to_corner, vertex_to_data):
        o = np.ascontiguousarray(opposite, dtype=np.uint32)
        c = np.ascontiguousarray(corner_to_vertex, dtype=np.uint32)
        d = np.ascontiguousarray(data_to_corner, dtype=np.uint32)
        v = np.ascontiguousarray(vertex_to_data, dtype=np.int32)
        # the library BORROWS the four arrays until the decode / upload call that consumes them returns
        # (include/dracob200.h): keep them alive with the batch
        self._borrowed = getattr(self, "_borrowed", {})
        self._borrowed[(k, dec)] = (o, c, d, v)
        N.check(N.lib().dcb_set_mesh_maps(self.h, k, dec, o.ctypes.data, c.ctypes.data, o.size, d.ctypes.data, d.size,
                                          v.ctypes.data, v.size))

    def set_output_order(self, points: bool):
        """DCB_ORDER_POINTS (points=True): attributes of Edgebreaker meshes come out as one row per point."""
        N.check(N.lib().dcb_set_output_order(self.h, N.DCB_ORDER_POINTS if points else N.DCB_ORDER_ENTRIES))
        self.point_order = bool(points)

    def set_face_output(self, on: bool):
        """DCB_FACES_ARENA (on=True): every mesh buffer's faces land in the output arena (face_info).  Set it before
        host_connectivity, so that the plain indices of sequential meshes are decoded on the GPU."""
        N.check(N.lib().dcb_set_face_output(self.h, N.DCB_FACES_ARENA if on else N.DCB_FACES_NONE))
        self.faces_in_arena = bool(on)

    def face_info(self, k):
        """Where buffer k's faces lie in the output arena (dcb_face_info; all zero without a faces region)."""
        fi = N.FaceInfo()
        N.check(N.lib().dcb_get_face_info(self.h, k, C.byref(fi)))
        return fi

    def set_mesh_faces(self, k, faces):
        """Faces (point ids) of Edgebreaker buffer k for point order; None: the NULL form (faces = corner_to_vertex
        of attributes decoder 0).  Borrowed by the library like the maps: kept alive with the batch."""
        self._borrowed = getattr(self, "_borrowed", {})
        if faces is None:
            self._borrowed[(k, "faces")] = None
            N.check(N.lib().dcb_set_mesh_faces(self.h, k, None, 0))
            return
        f = np.ascontiguousarray(faces, dtype=np.uint32).reshape(-1)
        if f.size % 3:
            raise ValueError("faces: 3 point ids per face")
        self._borrowed[(k, "faces")] = f
        N.check(N.lib().dcb_set_mesh_faces(self.h, k, f.ctypes.data if f.size else None, f.size // 3))

    def host_connectivity(self, k):
        """Decode the Edgebreaker connectivity of mesh buffer k on the host (dcb_host_connectivity)."""
        N.check(N.lib().dcb_host_connectivity(self.h, k))

    def faces(self, k):
        n = C.c_uint64(0)
        N.check(N.lib().dcb_mesh_faces(self.h, k, None, 0, C.byref(n)))
        f = np.zeros((n.value, 3), dtype=np.uint32)
        if n.value:
            N.check(N.lib().dcb_mesh_faces(self.h, k, f.ctypes.data, n.value, C.byref(n)))
        return f

    def mesh_map(self, k, attr_decoder, which):
        """which: 0 opposite, 1 corner_to_vertex, 2 data_to_corner (uint32), 3 vertex_to_data (int32)."""
        n = C.c_uint64(0)
        N.check(N.lib().dcb_mesh_map(self.h, k, attr_decoder, which, None, 0, C.byref(n)))
        m = np.zeros(n.value, dtype=np.uint32)
        if n.value:
            N.check(N.lib().dcb_mesh_map(self.h, k, attr_decoder, which, m.ctypes.data, n.value, C.byref(n)))
        return m.view(np.int32) if which == 3 else m

    def finish(self):
        N.check(N.lib().dcb_index_finish(self._dec.ctx if self._dec else None, self.h))


def index_only(buffers: Sequence) -> Batch:
    """Host indexing without a device (dcb_index with a NULL ctx): header-level inspection only."""
    return _index(None, buffers)


def _index(dec, buffers):
    arrs = [np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b, dtype=np.uint8)
            for b in buffers]
    n = len(arrs)
    ptrs = (C.c_void_p * max(n, 1))(*[a.ctypes.data if a.size else None for a in arrs])
    lens = (C.c_uint64 * max(n, 1))(*[a.size for a in arrs])
    h = C.c_void_p()
    N.check(N.lib().dcb_index(dec.ctx if dec else None, ptrs, lens, n, C.byref(h)))
    return Batch(dec, h, n, (arrs, ptrs, lens))


class DracoBatchDecoder:
    """GPU batch decoder.  `devices`: CUDA device ordinals (default: the current device)."""

    def __init__(self, devices: Optional[Sequence[int]] = None):
        self.ctx = C.c_void_p()
        if devices:
            ids = (C.c_int * len(devices))(*devices)
            rc = N.lib().dcb_create(ids, len(devices), C.byref(self.ctx))
        else:
            rc = N.lib().dcb_create(None, 0, C.byref(self.ctx))
        N.check(rc, "dcb_create")

    def close(self):
        if self.ctx:
            N.lib().dcb_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, dev_index, cuda_stream):
        N.check(N.lib().dcb_set_stream(self.ctx, dev_index, C.c_void_p(cuda_stream)))

    def set_limits(self, max_points_per_buffer=0, points_per_byte=4096):
        """Plausibility limits of one buffer (dcb_set_limits): a forged point count fails its own buffer."""
        N.check(N.lib().dcb_set_limits(self.ctx, max_points_per_buffer, points_per_byte))

    # ---- indexing ----
    def index(self, buffers: Sequence) -> Batch:
        return _index(self, buffers)

    def index_arena(self, arena: np.ndarray, offs: np.ndarray, lens: np.ndarray, arena_ptr: Optional[int] = None) -> Batch:
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        lens = np.ascontiguousarray(lens, dtype=np.uint64)
        h = C.c_void_p()
        ptr = arena_ptr if arena_ptr is not None else arena.ctypes.data
        N.check(N.lib().dcb_index_arena(self.ctx, ptr, offs.ctypes.data_as(C.POINTER(C.c_uint64)),
                                        lens.ctypes.data_as(C.POINTER(C.c_uint64)), offs.size, C.byref(h)))
        return Batch(self, h, int(offs.size), (arena, offs, lens))

    # ---- device phases ----
    def upload(self, batch: Batch):
        N.check(N.lib().dcb_upload(self.ctx, batch.h))

    def decode_resident(self, batch: Batch, dev_out: int = 0, dev_dbg: int = 0, flags: int = 0):
        N.check(N.lib().dcb_decode_resident(self.ctx, batch.h, C.c_void_p(dev_out), C.c_void_p(dev_dbg), flags))

    def download(self, batch: Batch, host_out: Optional[np.ndarray], host_dbg: Optional[np.ndarray] = None):
        N.check(N.lib().dcb_download(self.ctx, batch.h, host_out.ctypes.data if host_out is not None else None,
                                     host_dbg.ctypes.data if host_dbg is not None else None))

    def decode(self, batch: Batch, host_out: Optional[np.ndarray] = None, flags: int = 0, out_ptr: Optional[int] = None):
        """One call: H2D, kernels, D2H.  Returns (out arena, dbg arena or None)."""
        if host_out is None and out_ptr is None:
            host_out = np.empty(max(batch.out_bytes, 1), dtype=np.uint8)
        dbg = None
        if flags & (N.DCB_DUMP_SYMBOLS | N.DCB_DUMP_QINTS):
            dbg = np.zeros(max(batch.dbg_bytes, 1), dtype=np.uint8)
        N.check(N.lib().dcb_decode(self.ctx, batch.h, out_ptr if out_ptr is not None else host_out.ctypes.data,
                                   dbg.ctypes.data if dbg is not None else None, flags))
        return host_out, dbg

    def stats(self) -> N.LaunchStats:
        s = N.LaunchStats()
        N.check(N.lib().dcb_last_stats(self.ctx, C.byref(s)))
        return s

    # ---- the reference-shaped API ----
    def decode_batch(self, buffers: Sequence, point_order: bool = False, faces_in_arena: bool = False) -> List[Draco]:
        """DecodeBatch: one `Draco` per input buffer; a malformed buffer carries its status and no
        attributes (the reference would have thrown for that buffer alone).  point_order: attributes of
        Edgebreaker meshes hold one row per point, so that `values[faces]` is the mesh's triangle soup.
        faces_in_arena: the faces come out of the output arena (sequential plain indices decoded on the GPU);
        `Draco.faces` is then a view of it."""
        batch = self.index(buffers)
        try:
            if point_order:
                batch.set_output_order(True)
            if faces_in_arena:
                batch.set_face_output(True)
            meshes = [k for k in range(batch.n_bufs) if batch.buffer_info(k).needs_connectivity]
            for k in meshes:
                batch.host_connectivity(k)  # connectivity stays on the host (SURVEY 8f-1)
            if meshes:
                batch.finish()
            out, _ = self.decode(batch)
            return self.wrap(batch, out)
        finally:
            batch.free()

    def wrap(self, batch: Batch, out: np.ndarray) -> List[Draco]:
        res = []
        for k in range(batch.n_bufs):
            bi = batch.buffer_info(k)
            hdr = None
            if bi.status not in (-1, -2) or bi.version_major:
                hdr = DracoHeader(bi.version_major, bi.version_minor, bi.geometry_type, bi.encoder_method, bi.flags)
            d = Draco(header=hdr, status=bi.status, points_count=bi.n_points)
            if bi.status == 0 and bi.geometry_type == 1 and batch.faces_in_arena:
                fi = batch.face_info(k)
                f = out[fi.out_off: fi.out_off + fi.out_bytes].view(np.uint32).reshape(-1, 3)
                d.faces = f if fi.n_faces else None
            elif bi.status == 0 and bi.geometry_type == 1:
                f = batch.faces(k)
                d.faces = f if f.shape[0] else None  # None: the caller supplied the connectivity itself
            if bi.status == 0:
                for a in range(bi.n_attrs):
                    ai = batch.attr_info(k, a)
                    stride = ai.num_components * np.dtype(NP_DTYPES[ai.data_type]).itemsize
                    buf = out[ai.out_off: ai.out_off + ai.out_bytes]
                    pts = batch.point_order and bi.geometry_type == 1 and bi.encoder_method == 1
                    d.attributes.append(PointAttribute(ai.att_type, ai.data_type, ai.num_components, bool(ai.normalized),
                                                       ai.unique_id, stride, ai.n_entries, buf, ai, pts))
            res.append(d)
        return res
