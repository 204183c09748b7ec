"""NumPy statement of the point-order rule (MeshTraversalSequencer.UpdatePointToAttributeIndexMapping,
MeshTraversalSequencer.cs:33-51), independent of the library: for each corner c in increasing order,
map[faces[c]] = vertex_to_data[corner_to_vertex[c]]; the last corner of a point wins; -1: no corner."""
import numpy as np


def point_map(faces, corner_to_vertex, vertex_to_data, n_points):
    f = np.asarray(faces, dtype=np.int64).ravel()
    entry = np.asarray(vertex_to_data, dtype=np.int64)[np.asarray(corner_to_vertex, dtype=np.int64)]
    win = np.full(n_points, -1, dtype=np.int64)
    np.maximum.at(win, f, np.arange(f.size, dtype=np.int64))
    m = np.full(n_points, -1, dtype=np.int64)
    m[win >= 0] = entry[win[win >= 0]]
    return m


def gather_rows(entry_bytes, row_bytes, m):
    """Rows of an entry-order attribute (raw bytes) in point order; zero rows where m < 0."""
    rows = np.asarray(entry_bytes, dtype=np.uint8).reshape(-1, row_bytes)
    out = np.zeros((m.size, row_bytes), dtype=np.uint8)
    out[m >= 0] = rows[m[m >= 0]]
    return out.ravel()


def row_bytes(ai):
    size = {1: 1, 2: 1, 3: 2, 4: 2, 5: 4, 6: 4, 7: 8, 8: 8, 9: 4, 10: 8, 11: 1}[ai.data_type]
    return size * ai.num_components
