// draco_sharp_b200/csrc/dcb_kernels.h -- host-callable launchers of the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dcb_internal.h"

#define DCB_TAG_CHUNK 256u   // points per bit-offset checkpoint of a Tagged stream = one warp-chunk of par_post2_kernel
#define DCB_PAR_WARPS 8u     // par_post2_kernel: independent persistent warps per CTA
#define DCB_RING_BYTES 128u   // per-lane shared-memory ring of compressed bytes (rANS kernels)
// chain / consumer warp pairs (dcb_rans_pc.cu): shared memory of one pair beyond its lanes' tables
#define DCB_PC_STAGES 4u       // queue depth in groups
#define DCB_PC_ROW_BYTES 64u   // one queue row: symbol j of all 32 lanes, 2 bytes each
#define DCB_PC_CTL_BYTES 112u  // mbarriers full[4] empty[4] setup handoff filled + flag[4]
#define DCB_PC_HAND_BYTES 48u  // per-lane hand-over record
// bucket-record kernels (dcb_rans_rec.cu)
#define DCB_REC_HAND_BYTES 56u // per-lane hand-over record
#define DCB_REC_STAGES 2u      // queue depth in groups: the tables need the shared memory more than the queue does
#define DCB_REC_CTL_BYTES 64u  // mbarriers full[2] empty[2] setup handoff + flag[2]
struct PcGeom {
  uint32_t tab_bytes;    // table part of a pair's slice (worst-case alignment slack included)
  uint32_t slice_bytes;  // whole slice
  uint32_t q_off, ctl_off, hand_off;  // offsets inside the slice
  uint32_t fuse;         // raw kernel, direct slot LUT: the chain warp may keep the post-processing (fused_direct_loop)
};

// device arenas of one shard
struct DevArenas {
  const uint8_t *in;  // compressed buffers, each on a 16-byte boundary
  uint8_t *out;       // attribute outputs, each on a 128-byte boundary
  uint8_t *dbg;       // DCB_DUMP_*: int32 per portable value
  uint8_t *aux;       // scratch: corrections / tags / parallelogram dependencies
  uint8_t *tab;       // scratch: probability tables that do not fit shared memory
  const uint8_t *maps;  // mesh connectivity maps
};

uint32_t dcb_rans_smem_bytes(const RansLaunch &p, bool table_global);
// Raw-scheme rANS decode fused with inverse prediction + transform + store; one stream per lane.
cudaError_t dcb_launch_rans_raw(const RansLaunch &p, int ncp, bool wide, bool table_global, const DevArenas &a,
                                cudaStream_t st);
// the same two kernels as chain / consumer warp pairs (u16 tables in shared memory only)
PcGeom dcb_pc_geom(const RansLaunch &p, uint32_t syms_per_group);
uint32_t dcb_rans_pc_smem_bytes(const RansLaunch &p, uint32_t syms_per_group);
cudaError_t dcb_launch_rans_raw_pc(const RansLaunch &p, int ncp, const DevArenas &a, cudaStream_t st);
cudaError_t dcb_launch_rans_tag_pc(const RansLaunch &p, const DevArenas &a, cudaStream_t st);
// bucket-record tables (dcb_rans_rec.cu): one dependent shared-memory access per symbol; warp pairs; RansLaunch::rec_ka / rec_bytes
uint32_t dcb_rans_rec_smem_bytes(const RansLaunch &p, uint32_t syms_per_group);
cudaError_t dcb_launch_rans_raw_rec(const RansLaunch &p, int ncp, const DevArenas &a, cudaStream_t st);
cudaError_t dcb_launch_rans_tag_rec(const RansLaunch &p, const DevArenas &a, cudaStream_t st);
// tag stream of Tagged attributes; one stream per lane
cudaError_t dcb_launch_rans_tag(const RansLaunch &p, const DevArenas &a, cudaStream_t st);
cudaError_t dcb_launch_resolve(const DevArenas &a, BufWalk *d_walks, const uint32_t *d_list, uint32_t n,
                               StreamDesc *d_streams, cudaStream_t st);
cudaError_t dcb_launch_serial_post(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, int ncp, uint32_t dump,
                                   uint32_t only_irregular, const DevArenas &a, cudaStream_t st);
// point-parallel path behind Tagged / uncompressed sources (recon none or delta + wrap; corrections of parallelogram /
// octahedral streams go to the int32 scratch).  Persistent warps pull runs of `run_len` chunks from *d_ticket;
// d_run_prefix[i] = runs in front of stream d_order[i] (n + 1 values).
uint32_t dcb_par_post_smem_bytes(int ncp);
// run length (chunks) and runs per ticket for a launch: whole streams when there are enough of them, else single chunks
void dcb_par_post_plan(uint32_t n_streams, uint64_t total_chunks, uint32_t max_chunks, bool any_delta, uint32_t num_sms, int ncp,
                       uint32_t share,
                       uint32_t *run_len, uint32_t *claim);
// n_rounds != 0: chunk-sized runs ticketed round by round; d_run_prefix then has n_rounds + 1 entries (runs in front of round r)
cudaError_t dcb_launch_par_post(StreamDesc *d_streams, const uint32_t *d_order, const uint32_t *d_run_prefix, uint32_t n,
                                uint32_t total_runs, uint32_t run_len, uint32_t claim, uint32_t n_rounds, unsigned int *d_ticket, uint32_t num_sms,
                                int ncp, uint32_t dump, uint32_t epoch, const DevArenas &a, cudaStream_t st);
cudaError_t dcb_launch_para(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, int ncp, uint32_t max_entries,
                            uint32_t dump, const DevArenas &a, cudaStream_t st);
// MeshPredictionSchemeConstrainedMultiParallelogramDecoder (dcb_cmp.cu): cmp_flags_kernel (rABS crease flags, one warp per
// context; needs the bitstream only) | cmp_deps_kernel (point-parallel) + cmp_chain_kernel (one warp per stream)
cudaError_t dcb_launch_cmp_flags(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, const DevArenas &a, cudaStream_t st);
cudaError_t dcb_launch_cmp_deps(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t max_entries, const DevArenas &a,
                                cudaStream_t st);
cudaError_t dcb_launch_cmp(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, int ncp, uint32_t dump, const DevArenas &a,
                           cudaStream_t st);
// MeshPredictionSchemeGeometricNormalDecoder (dcb_geonormal.cu): geo_flips_kernel (rABS flip bits, one warp per stream; needs
// the bitstream only) | geo_normal_kernel (point-parallel: prediction from the parent's decoded positions, octahedron transform, unit vectors)
cudaError_t dcb_launch_geo_flips(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, const DevArenas &a, cudaStream_t st);
cudaError_t dcb_launch_geo_normal(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t max_entries, uint32_t dump,
                                  const DevArenas &a, cudaStream_t st);
// MeshPredictionSchemeTexCoordsPortableDecoder (dcb_texcoord.cu): tex_prep_kernel (point-parallel) + tex_chain_kernel
// (one warp per stream); the parent position streams must have been through dcb_launch_para on the same stream
cudaError_t dcb_launch_tex(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t max_entries, uint32_t dump,
                           const DevArenas &a, cudaStream_t st);
// integer attributes with more than 4 components (run-time component count): reconstruction + narrowing store, one lane per stream
cudaError_t dcb_launch_wide_post(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t dump, const DevArenas &a,
                                 cudaStream_t st);
cudaError_t dcb_launch_oct_chain(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t dump,
                                 const DevArenas &a, cudaStream_t st);
cudaError_t dcb_launch_oct_unit(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t max_entries,
                                const DevArenas &a, cudaStream_t st);
cudaError_t dcb_launch_copy(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint64_t max_bytes,
                            const DevArenas &a, cudaStream_t st);

// ---- point order (DCB_ORDER_POINTS, dcb_points.cu) ----
// MeshTraversalSequencer.UpdatePointToAttributeIndexMapping: for each corner c of attributes decoder d,
// map_d[faces[c]] = vertex_to_data_d[corner_to_vertex_d[c]]; the last corner of a point wins.
#define DCB_POINT_NONE 0xFFFFFFFFu  // map value of a point no corner references: its rows are zero
struct PointMapJob {               // one (Edgebreaker buffer, attributes decoder)
  uint64_t faces_off;              // maps arena: point id per corner (explicit faces, or corner_to_vertex of decoder 0)
  uint64_t c2v_off, v2d_off;       // maps arena: the decoder's corner_to_vertex and vertex_to_data
  uint64_t map_off;                // point-map region, in u32: winning corner + 1, then the entry of each point
  uint32_t n_corners, n_points, n_vertices, n_entries;
  uint32_t status_si;              // stream that carries the buffer's DCB_ERR_MAPS
  uint32_t pad_;
};
struct PointGatherJob {            // one attribute of a point-order shard
  uint64_t src_off;                // entry-order staging
  uint64_t dst_off;                // output arena
  uint64_t map_off;                // point-map region (u32), ~0ull: identity rows (point clouds, sequential meshes)
  uint32_t rows, row_bytes;
  uint32_t st_first, st_count;     // the buffer's streams: a buffer with a failed stream is not gathered
  uint32_t vec_shift;              // log2 of the copy unit (16, 8, 4, 2 or 1 bytes; divides row_bytes)
  uint32_t pad_;
};
struct PointStage {
  const PointMapJob *maps;         // n_maps jobs; corner_prefix / point_prefix: n_maps + 1 running sums
  const uint64_t *corner_prefix, *point_prefix;
  uint32_t n_maps;
  const PointGatherJob *gathers;   // n_gathers jobs; unit_prefix: n_gathers + 1 running sums of rows * units per row
  const uint64_t *unit_prefix;
  uint32_t n_gathers;
  uint32_t *pmap;                  // point-map region (zeroed by the launcher before the corner pass)
  uint64_t pmap_words;             // = point_prefix[n_maps]
  uint64_t total_corners, total_units;  // = corner_prefix[n_maps], unit_prefix[n_gathers] (grid sizes)
  const uint8_t *stage;            // entry-order outputs of the shard's kernels
};
// point_win_kernel (one thread per corner) | point_resolve_kernel (one thread per point) | point_gather_kernel (one thread
// per copy unit of every row of every attribute), on `st`
cudaError_t dcb_launch_point_stage(const PointStage &p, StreamDesc *d_streams, const DevArenas &a, uint32_t num_sms,
                                   cudaStream_t st);

// ---- faces in the output arena (DCB_FACES_ARENA, dcb_faces.cu) ----
struct FaceJob {                   // the faces of one mesh buffer
  uint64_t src_off;                // first index byte: input arena (sequential plain indices) or maps arena (u32 faces)
  uint64_t dst_off;                // faces region in the output arena (128-byte aligned)
  uint64_t n_idx;                  // 3 * n_faces
  uint64_t n_bytes;                // varint: bytes of the index run
  uint64_t ckpt_off;               // varint: first checkpoint of the job (FaceStage::ckpt)
  uint32_t width;                  // bytes per index: 1, 2 or 4; 0 = varint
  uint32_t from_maps;              // 1: src_off is in the maps arena
  uint32_t stream;                 // Raw index differences: the shard-wide index of their rANS stream (symbols at its aux_off)
  uint32_t pad_;
};
struct FaceStage {
  const FaceJob *plain;            // fixed-width jobs; unit_prefix: n_plain + 1 running sums of ceil(n_idx / 4)
  const uint64_t *unit_prefix;
  uint32_t n_plain;
  const FaceJob *varint;           // varint jobs; chunk_prefix: n_varint + 1 running sums of their DCB_VARINT_CHUNK-byte chunks
  const uint64_t *chunk_prefix;
  uint32_t n_varint;
  const uint64_t *ckpt;            // per chunk: indices that end in front of it (located by the host)
  uint64_t total_units, total_chunks;  // = unit_prefix[n_plain], chunk_prefix[n_varint] (grid sizes)
  // Raw index differences (method 0): the rANS kernels leave the symbols in the int32 scratch; three passes over
  // DCB_INDEX_CHUNK-index chunks turn them into indices
  const FaceJob *index;            // index_prefix: n_index + 1 running sums of their chunks
  const uint64_t *index_prefix;
  uint32_t n_index;
  uint64_t total_index_chunks;
  int64_t *chunk_sum, *chunk_min, *chunk_max;  // per chunk: sum of its steps (then the index in front of it), extreme prefixes
  int32_t *status;                 // per index job: DCB_ERR_CONNECTIVITY or the failure of its rANS stream
};
#define DCB_INDEX_CHUNK 4096u
// seq_plain_kernel (one thread per 4 indices of every fixed-width job: widen to u32) | seq_varint_kernel (one CTA per
// chunk of a varint run: terminator bytes, their ordinals by a block scan from the chunk's checkpoint, values assembled
// backwards by the terminator's thread), on `st`
// seq_index_sum_kernel | seq_index_base_kernel | seq_index_store_kernel: Raw index differences (sign-magnitude steps,
// symbol >> 1, negative when bit 0 is set) -> inclusive int64 scan per buffer (chunk sums, then one thread per buffer over
// its chunks, then the chunks again) with the range checks of dcb_host_sequential (0 <= index <= INT32_MAX)
cudaError_t dcb_launch_faces(const FaceStage &p, const StreamDesc *d_streams, const DevArenas &a, uint32_t num_sms, cudaStream_t st);
