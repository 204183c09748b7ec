// draco_sharp_b200/csrc/dcb_points.cu -- attributes of Edgebreaker meshes in point order (DCB_ORDER_POINTS).
//
// The decode kernels write every attribute in entry order: the unique values in the order the depth-first traversal
// encoded them.  A mesh's faces index points.  The reference joins the two in MeshTraversalSequencer
// .UpdatePointToAttributeIndexMapping (MeshTraversalSequencer.cs:33-51): for each attributes decoder d and each corner c
// in increasing order
//     map_d[faces[c]] = vertex_to_data_d[corner_to_vertex_d[c]]
// so when two corners of one point disagree the later corner wins.  Three point-parallel passes reproduce that:
//   point_win_kernel      one thread per corner: bound checks of the point and vertex ids, winning corner per point
//                         with an integer max (red.global.max: the highest corner wins whatever order the writes land in)
//   point_resolve_kernel  one thread per point: winning corner -> vertex -> entry, bound check of the entry
//   point_gather_kernel   one thread per copy unit (16, 8, 4, 2 or 1 bytes) of each output row: row p of an attribute
//                         is row map_d[p] of its entry-order staging; unreferenced points get zero rows
// Malformed maps become DCB_ERR_MAPS on the buffer's first stream (as para_deps_kernel reports them); a buffer with a
// failed stream is not gathered.  Product code: nothing here touches oracle/.
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>

#include "dcb_internal.h"
#include "dcb_jobs.cuh"
#include "dcb_kernels.h"

namespace {

constexpr uint32_t kThreads = 256;
constexpr uint32_t kPerThread = 4;
constexpr uint32_t kTile = kThreads * kPerThread;  // consecutive elements of one block iteration

__device__ __forceinline__ void fail_maps(StreamDesc *streams, uint32_t si) {
  atomicCAS(&streams[si].status, (int32_t)DCB_OK, (int32_t)DCB_ERR_MAPS);
}

__global__ void __launch_bounds__(kThreads) point_win_kernel(PointStage p, StreamDesc *streams, const uint8_t *__restrict__ maps) {
  dcb_for_each_element<kThreads, kPerThread>(p.corner_prefix, p.n_maps, [&](uint32_t j, uint64_t ci) {
    const PointMapJob &m = p.maps[j];
    const uint32_t c = (uint32_t)ci;
    const uint32_t pt = reinterpret_cast<const uint32_t *>(maps + m.faces_off)[c];
    const uint32_t v = reinterpret_cast<const uint32_t *>(maps + m.c2v_off)[c];
    if (pt >= m.n_points || v >= m.n_vertices) {
      fail_maps(streams, m.status_si);
      return;
    }
    atomicMax(p.pmap + m.map_off + pt, c + 1u);  // n_corners <= 2^32 - 1: c + 1 never wraps; 0 = no corner
  });
}

__global__ void __launch_bounds__(kThreads) point_resolve_kernel(PointStage p, StreamDesc *streams, const uint8_t *__restrict__ maps) {
  dcb_for_each_element<kThreads, kPerThread>(p.point_prefix, p.n_maps, [&](uint32_t j, uint64_t pi) {
    const PointMapJob &m = p.maps[j];
    uint32_t *slot = p.pmap + m.map_off + pi;
    const uint32_t win = *slot;
    uint32_t e = DCB_POINT_NONE;
    if (win != 0) {
      const uint32_t v = reinterpret_cast<const uint32_t *>(maps + m.c2v_off)[win - 1u];  // checked by the corner pass
      const int32_t ev = reinterpret_cast<const int32_t *>(maps + m.v2d_off)[v];
      if (ev < 0 || (uint32_t)ev >= m.n_entries) fail_maps(streams, m.status_si);
      else e = (uint32_t)ev;
    }
    *slot = e;
  });
}

template <typename T>
__device__ __forceinline__ void copy_unit(uint8_t *dst, const uint8_t *src) {
  if (src) *reinterpret_cast<T *>(dst) = *reinterpret_cast<const T *>(src);
  else *reinterpret_cast<T *>(dst) = T{};
}

__global__ void __launch_bounds__(kThreads) point_gather_kernel(PointStage p, const StreamDesc *streams, uint8_t *__restrict__ out) {
  uint32_t cur = 0xFFFFFFFFu;
  bool ok = false;
  dcb_for_each_element<kThreads, kPerThread>(p.unit_prefix, p.n_gathers, [&](uint32_t j, uint64_t u) {
    const PointGatherJob &g = p.gathers[j];
    if (j != cur) {  // a thread meets few jobs: check the buffer's statuses once per job
      cur = j;
      ok = true;
      for (uint32_t s = 0; s < g.st_count; ++s) ok = ok && streams[g.st_first + s].status == DCB_OK;
    }
    if (!ok) return;
    const uint32_t units = g.row_bytes >> g.vec_shift;
    const uint64_t r = u / units;
    const uint64_t w = (u - r * units) << g.vec_shift;
    const uint32_t e = g.map_off == ~0ull ? (uint32_t)r : p.pmap[g.map_off + r];
    uint8_t *dst = out + g.dst_off + r * g.row_bytes + w;
    const uint8_t *src = e == DCB_POINT_NONE ? nullptr : p.stage + g.src_off + (uint64_t)e * g.row_bytes + w;
    switch (g.vec_shift) {
      case 4: copy_unit<uint4>(dst, src); break;
      case 3: copy_unit<uint2>(dst, src); break;
      case 2: copy_unit<uint32_t>(dst, src); break;
      case 1: copy_unit<uint16_t>(dst, src); break;
      default: copy_unit<uint8_t>(dst, src); break;
    }
  });
}

uint32_t grid_for(uint64_t total, uint32_t num_sms) {
  const uint64_t tiles = (total + kTile - 1) / kTile;
  return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(tiles, (uint64_t)num_sms * 8));
}

}  // namespace

cudaError_t dcb_launch_point_stage(const PointStage &p, StreamDesc *d_streams, const DevArenas &a, uint32_t num_sms,
                                   cudaStream_t st) {
  if (p.pmap_words) {
    cudaError_t e = cudaMemsetAsync(p.pmap, 0, p.pmap_words * 4, st);
    if (e != cudaSuccess) return e;
  }
  if (p.total_corners) point_win_kernel<<<grid_for(p.total_corners, num_sms), kThreads, 0, st>>>(p, d_streams, a.maps);
  if (p.pmap_words) point_resolve_kernel<<<grid_for(p.pmap_words, num_sms), kThreads, 0, st>>>(p, d_streams, a.maps);
  if (p.total_units) point_gather_kernel<<<grid_for(p.total_units, num_sms), kThreads, 0, st>>>(p, d_streams, a.out);
  return cudaGetLastError();
}
