// draco_sharp_b200/csrc/dcb_mesh_host.h -- host Edgebreaker connectivity helper (see dcb_mesh_host.cu)
#pragma once
#include <stdint.h>

#include <vector>

struct DcbHostMaps {
  std::vector<uint32_t> opposite, corner_to_vertex, data_to_corner;
  std::vector<int32_t> vertex_to_data;
};

// Decodes the Edgebreaker connectivity of one mesh buffer on the CPU.  Outputs where ATTRIBUTES starts, the
// point count, one set of maps per attributes decoder and (optionally) the faces as 3 point ids each.
int dcb_host_edgebreaker(const uint8_t *buf, uint64_t len, uint64_t conn_off, uint64_t *attr_section_off,
                         uint32_t *n_points, std::vector<DcbHostMaps> *maps, std::vector<uint32_t> *faces);

// Indices of a sequential mesh, located but not decoded (DCB_FACES_ARENA: the GPU decodes them): plain indices
// (connectivity method 1) or a Raw symbol stream of index differences (method 0)
struct DcbSeqIndexLoc {
  bool located = false;
  uint64_t n_idx = 0;          // 3 * n_faces
  uint64_t off = 0, bytes = 0; // first index byte inside the buffer (Raw: the RANS_TABLE), bytes up to the end of the indices
  int width = 0;               // 1, 2, 4; 0 = varint; -1 = Raw symbols
  int mbl = 0;                 // Raw: max_bit_length
  std::vector<uint64_t> ckpt;  // varint: indices that end in front of each DCB_VARINT_CHUNK-byte chunk of the run
};

// Decodes the connectivity of a SEQUENTIAL mesh buffer (MeshSequentialDecoder.cs:8-118) on the CPU: where ATTRIBUTES
// starts, the point count, the faces as 3 point ids each.  Its attributes need no maps.  loc != NULL: plain indices and
// Raw index streams are located into *loc instead, after the same checks with the same statuses, and *faces stays
// empty; a Tagged index stream is decoded (its bit area has no length prefix: SymbolDecoding.cs:37-49).
int dcb_host_sequential(const uint8_t *buf, uint64_t len, uint64_t conn_off, uint64_t *attr_section_off, uint32_t *n_points,
                        std::vector<uint32_t> *faces, DcbSeqIndexLoc *loc = nullptr);
