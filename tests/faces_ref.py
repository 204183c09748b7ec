"""Sequential meshes for the faces-in-the-arena tests (DCB_FACES_ARENA): grids and long strips, written by drc_writer, over
every index coding of MeshSequentialDecoder.cs: entropy-coded differences (Raw, Tagged) and plain indices of 1, 2, varint
and 4 bytes."""
import numpy as np

import drc_writer as W


def grid_faces(w, h):
    f = []
    for y in range(h - 1):
        for x in range(w - 1):
            a = y * w + x
            f += [(a, a + 1, a + w), (a + 1, a + w + 1, a + w)]
    return f


def strip_faces(n_points, n_tri):
    """n_tri triangles of a strip over the highest point ids: large point counts (index widths) with few faces."""
    base = n_points - n_tri - 2
    return [(base + i, base + i + 1 + (i & 1), base + i + 2 - (i & 1)) for i in range(n_tri)]


def attrs(n_points, seed):
    rng = np.random.default_rng(seed)
    corr = rng.integers(-20, 21, size=n_points * 3)
    return [dict(att_type=0, data_type=9, nc=3, seq_type=2, portable=W.portable_int(corr, 3, 0, 1, "raw", W.wrap_data(0, 4095)),
                 xform=W.quant_params([0.0, 1.0, 2.0], 8.0, 12))]


def mesh(faces, n_points, method, scheme="raw", with_attrs=True, seed=0):
    a = attrs(n_points, seed) if with_attrs else []
    return np.frombuffer(W.sequential_mesh(faces, n_points, a, method, scheme), dtype=np.uint8)


def index_width(n_points):
    """bytes per plain index (method 1), 0 = varint"""
    return 1 if n_points < 256 else 2 if n_points < (1 << 16) else 0 if n_points < (1 << 21) else 4
