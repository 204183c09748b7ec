// draco_sharp_b200/csrc/dcb_api.cu -- C ABI of libdracob200.so (include/dracob200.h): host indexer,
// launch planner and the decode driver.  Host code only; the kernels are in dcb_kernels.cu.
//
// Host-side reference semantics restated here (src/Draco/IO/...):
//   header             DracoDecoder.cs:44-64 (magic, version, geometry type, method, flags)
//   metadata (skipped) Metadata/MetadataDecoder.cs:5-49
//   ATTRIBUTES         ConnectivityDecoder.cs:16-44, Mesh/MeshEdgeBreakerDecoder.cs:642-662 (DEC_ID),
//                      Attributes/AttributesDecoder.cs:19-63 (DEC_DATA),
//                      Attributes/SequentialAttributeDecodersController.cs:16-27 (decoder type bytes)
//   entry counts       Attributes/LinearSequencer.cs:7-13 (num_points), MeshAttributeIndicesEncodingObserver.cs:14-21
// The payload walk itself is dcb_walk.h.  There is NO CPU decode path in this library.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <chrono>
#include <thread>
#include <mutex>
#include <memory>
#include <string>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <new>
#include <tuple>
#include <vector>

#include "dcb_internal.h"
#include "dcb_kernels.h"
#include "dcb_mesh_host.h"
#include "dcb_walk.h"

namespace {

constexpr uint64_t kFrontPad = 256;    // bytes before the first buffer in the device input arena
constexpr uint64_t kBackPad = 64;      // bytes after the last one (16-byte window loads may overrun)
constexpr uint32_t kNumSMsDefault = 148;
constexpr uint32_t kSmemPerSM = 227 * 1024;
constexpr uint32_t kSmemPerCtaReserve = 1024;
constexpr uint64_t kTabArenaBudget = 1ull << 30;
constexpr uint64_t kDefaultPointsPerByte = 4096;

inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// experiment / test switches, read once per process (never per stream or per decode)
struct EnvFlags {
  bool debug_plan, debug_timing, lutb_full, rans_pc, no_direct, no_fast_tagged, no_threads;
  int rec_ka;
  bool no_rec, split;
  EnvFlags() {
    debug_plan = getenv("DCB_DEBUG_PLAN") != nullptr;
    debug_timing = getenv("DCB_DEBUG_TIMING") != nullptr;
    lutb_full = getenv("DCB_LUTB_FULL") != nullptr;
    rans_pc = getenv("DCB_RANS_PC") != nullptr;      // chain / consumer warp pairs for every u16 group (experiments)
    no_direct = getenv("DCB_NO_DIRECT") != nullptr;  // never plan the direct slot LUT
    no_threads = getenv("DCB_NO_THREADS") != nullptr;          // multi-device decodes on the calling thread only
    no_fast_tagged = getenv("DCB_NO_FAST_TAGGED") != nullptr;  // always fetch the resumed walks before classifying
    no_rec = getenv("DCB_REC") == nullptr;                               // the bucket-record kernels are opt-in (DCB_REC=1): measured
                                                                         // slower than the fused kernel at full residency (DESIGN 3.1)
    split = getenv("DCB_SPLIT") != nullptr;                              // warp-pair kernels: consumers on their own sub-partition
    rec_ka = getenv("DCB_REC_KA") ? atoi(getenv("DCB_REC_KA")) : 0;     // force their wide-region bucket size (experiments)
  }
};
const EnvFlags &env_flags() {
  static const EnvFlags f;
  return f;
}

// Device-memory cache of a context: the big per-batch arenas (input, output, scratch, maps) are returned here when a
// batch is freed and reused by the next one -- a cudaMalloc / cudaFree pair of 15 GB costs 10-100 ms, more than the
// kernels of the batch.  Blocks are handed out when they are at most twice the size asked for; the cache is capped.
struct PoolBlock {
  void *p;
  uint64_t bytes;
  int device;
};
struct DevPool {
  std::mutex mu;  // decode threads of different devices share the context's cache
  std::vector<PoolBlock> free_blocks;
  std::vector<PoolBlock> free_pinned;  // page-locked staging buffers (device = -1)
  uint64_t cached = 0;
};
constexpr uint64_t kPoolCap = 96ull << 30;
constexpr uint64_t kPoolMin = 0;  // every arena goes through the cache: a small batch pays for each cudaMalloc / cudaFree too

// Connectivity maps of one attributes decoder.  The arrays are BORROWED from the caller (dcb_set_mesh_maps: they must
// stay valid until the decode / upload call that consumes them returns) -- 56 bytes per vertex that are only read once,
// by the H2D copy; the library's own host helper (dcb_host_connectivity) parks its results in `own`.
struct MeshMapsHost {
  const uint32_t *opposite = nullptr, *corner_to_vertex = nullptr, *data_to_corner = nullptr;
  const int32_t *vertex_to_data = nullptr;
  uint64_t n_corners = 0, n_entries = 0, n_vertices = 0;
  std::shared_ptr<DcbHostMaps> own;
  bool set = false;
  uint64_t dev_off[4] = {0, 0, 0, 0};
  uint64_t bytes() const { return 4ull * (2 * n_corners + n_entries + n_vertices); }
};

struct BufRec {
  const uint8_t *src = nullptr;
  uint64_t len = 0;
  uint64_t arena_off = 0;  // inside the shard's device input arena
  int shard = 0;
  int local = 0;           // index inside the shard
  dcb_buffer_info info{};
  bool is_eb = false;
  std::vector<MeshMapsHost> maps;  // per attributes decoder
  std::vector<uint32_t> faces;     // dcb_host_connectivity: 3 point ids per face
  uint64_t conn_off = 0;           // meshes: first byte after header + metadata
  std::vector<uint32_t> dec_entries;
  // point order (Edgebreaker): faces set by dcb_set_mesh_faces / dcb_host_connectivity -- BORROWED like the maps, or
  // the NULL form (point ids = corner_to_vertex of decoder 0)
  const uint32_t *pt_faces = nullptr;
  uint64_t pt_n_faces = 0;
  bool pt_faces_set = false;
  bool pt_failed = false;          // the status is the point-order face check's verdict (undone when indexing reruns)
  uint64_t faces_dev_off = 0;      // explicit faces inside the shard's maps arena
  // faces in the output arena (DCB_FACES_ARENA).  pt_faces / pt_n_faces also carry the host-decoded faces of a sequential
  // mesh there: they travel with the maps like an Edgebreaker buffer's explicit faces.
  DcbSeqIndexLoc seq_loc;          // sequential, plain indices: located by dcb_host_connectivity, decoded on the GPU
  int32_t face_src = 0;            // dcb_face_info.source of the current layout
  int32_t idx_job = -1;            // Raw index differences decoded on the GPU: the buffer's slot in Shard::h_fstatus
  uint64_t n_faces = 0, face_off = 0;  // face_off: shard-local offset of the faces region
};

struct Stage {                 // the streams of one stage's launch
  std::vector<uint32_t> order;
  uint64_t order_off = 0;      // offset (in uint32) inside the shard's device order array
  uint32_t max_entries = 0;
  uint64_t max_bytes = 0;
};

struct Group : Stage {    // one rANS launch (or a few, for global tables) and its geometry
  bool tag;               // the tags of Tagged streams (16 symbols per step), not the values of Raw ones
  int ncp;
  bool wide, table_global;
  uint32_t compact, prec_bits, entries, exc, lut_shift, lut_bytes, lutb_bytes, ent_bytes, lanes, zig, mode;
  uint32_t pairs;         // chain/consumer warp pairs per CTA (0: the single-warp kernels of dcb_kernels.cu)
  uint32_t direct;        // direct slot LUT (warp-pair kernels)
  uint64_t total_symbols;
  // earliest / latest 128-slot block (over the group's streams) holding the first entry narrower than 2^k slots
  uint32_t nb_min[8], nb_max[8];
  bool nb_any;
  // bucket-record kernels (dcb_rans_rec.cu): largest table need over the group's streams per candidate bucket size
  // (8-byte units, 0xFFFF = some stream's table does not have the shape), value slots over ALL streams, and the plan
  uint32_t rec_max[4], exc_all;
  uint32_t rec_ka, rec_bytes;  // rec_ka != 0: the group runs on the bucket-record kernels
  uint32_t split;              // warp-pair kernels: chain warps on sub-partitions 0..2, consumers on sub-partition 3
  bool no_direct;              // a machine-filling group runs in the same step: keep this one's shared memory small
  bool force_single_warp;      // wide attributes: only the fused single-warp kernel knows to decode n * nc symbols
  void note_table(const StreamDesc &s) {
    for (int k = 1; k <= 7; ++k) {
      nb_min[k] = nb_any ? std::min<uint32_t>(nb_min[k], s.narrow_blk[k]) : s.narrow_blk[k];
      nb_max[k] = nb_any ? std::max<uint32_t>(nb_max[k], s.narrow_blk[k]) : s.narrow_blk[k];
    }
    for (int j = 0; j < 4; ++j) rec_max[j] = nb_any ? std::max<uint32_t>(rec_max[j], s.rec_need[j]) : s.rec_need[j];
    exc_all = std::max(exc_all, s.n_active - std::min(s.n_active, s.dense_prefix));
    nb_any = true;
  }
};

// The launches of one decode of a shard after its tag rounds, planned on the host from the ready streams (plan_shard):
// built without a CUDA call, then issued by decode_shard.  Stage arrays are indexed by component count 1..4.
struct ShardPlan {
  std::vector<Group> raw;  // Raw rANS groups, in RawKey order
  int dom = -1;            // raw[dom]: the group with the most symbols (statistics and kernel name of the decode)
  Stage post[5], para[5], cmp[5], par[5], copy, octs, octc, tex, geo, wide;
  struct ParPost {         // par_post2_kernel of par[n]: per group the run prefix of its streams and one ticket word
    bool delta = false;
    uint32_t run_len = 1, claim = 1, rounds = 0;
    std::vector<uint32_t> runs;
    uint64_t runs_off = 0;  // offset (in uint32) of `runs` inside the device order array
  } pp[5];
  bool has_para = false;        // mesh kernels validate the caller's maps on the device
  bool side_followers = false;  // oct_chain / oct_unit run next to the rANS kernels of other groups
  std::vector<uint32_t> order;  // the device order array: every stage list, then the runs
  bool flag_kernels() const {   // crease flags / flip bits of the 8f-3 predictors
    bool any = !geo.order.empty();
    for (int n = 1; n <= 4; ++n) any = any || !cmp[n].order.empty();
    return any;
  }
};

struct Shard {
  bool direct = false;  // the shard's buffers are one 16-byte aligned range of the caller's arena: upload it as is
  uint64_t direct_lo = 0, direct_hi = 0;
  int share = 1;        // shards of this batch living on the same physical device (pipeline slices)
  bool arena_pending = false;
  bool maps_pending = false;  // mesh maps allocated on the device, not copied yet
  std::shared_ptr<DevPool> pool;  // the owning context's cache (outlives the context if batches are freed late)
  uint64_t cap_in = 0, cap_out = 0, cap_aux = 0, cap_maps = 0, cap_stage = 0, cap_streams = 0, cap_walks = 0, cap_order = 0;
  int device = 0;
  std::vector<int> bufs;
  std::vector<StreamDesc> streams, streams0;
  std::vector<BufWalk> walks, walks0;
  std::vector<uint8_t> tags_launched;
  PointStage pstage{};         // point order: device job tables (plan_points)
  uint64_t in_bytes = 0, out_bytes = 0, dbg_bytes = 0, aux_bytes = 0, maps_bytes = 0;
  uint64_t out_base = 0, dbg_base = 0;  // offset of this shard inside the batch-wide host arenas
  // device
  uint8_t *d_in = nullptr, *d_out = nullptr, *d_dbg = nullptr, *d_aux = nullptr, *d_tab = nullptr, *d_maps = nullptr;
  uint64_t tab_cap = 0, dbg_cap = 0;
  StreamDesc *d_streams = nullptr;
  BufWalk *d_walks = nullptr;
  uint32_t *d_order = nullptr;
  uint64_t order_cap = 0;
  uint8_t *h_stage = nullptr;  // pinned staging for the packed input
  uint8_t *h_maps = nullptr;   // pinned staging for large sets of (borrowed, pageable) mesh maps
  uint64_t cap_hmaps = 0;
  uint8_t *h_desc = nullptr;   // pinned staging: device-updated stream descriptors + walks travel back without blocking
  uint64_t cap_hdesc = 0;
  bool desc_pending = false;   // h_desc holds a copy-back that absorb_descs folds into streams / walks after the sync
  ShardPlan plan;              // of the decode in flight (its order array is the source of an asynchronous upload)
  uint32_t epoch = 0;          // tags the look-back words of par_post2_kernel (30 bits, never 0): no clearing between decodes
  bool uploaded = false, dirty = true, own_out = false;
  uint8_t *ext_out = nullptr, *ext_dbg = nullptr;
  // output arena layout per stream: where the attribute lands for the caller.  Entry order: the stream's own out_off /
  // out_bytes.  A point-order shard (pts: it holds an Edgebreaker buffer in DCB_ORDER_POINTS) runs its kernels into an
  // entry-order staging arena laid out by out_off (stage_bytes, at the front of d_pts) and the point stage fills the
  // output arena from it.
  std::vector<uint64_t> fin_off, fin_bytes;
  bool pts = false;
  uint64_t stage_bytes = 0;
  uint8_t *d_pts = nullptr;    // staging | point maps | job tables
  uint64_t cap_pts = 0;
  std::vector<uint8_t> pts_tables;  // host copy of the job tables (source of the asynchronous upload)
  // DCB_FACES_ARENA: job tables of the faces stage (dcb_faces.cu) and their host copy
  FaceStage fstage{};
  uint8_t *d_faces = nullptr;
  uint64_t cap_faces = 0;
  std::vector<uint8_t> faces_tables;
  // Raw index differences of sequential meshes: one rANS stream each, appended to `streams` behind the attributes of
  // all buffers (from idx_first on; no buffer's walk covers them); their per-buffer verdicts come back in h_fstatus
  uint32_t idx_first = ~0u;
  int32_t *h_fstatus = nullptr;
  uint64_t cap_hfstatus = 0;
};

}  // namespace

struct dcb_ctx {
  std::vector<int> devices;
  std::vector<cudaStream_t> streams;
  std::vector<bool> own_stream;
  std::vector<int> num_sms;
  // side streams: independent rANS groups of one decode run concurrently (their CTAs share the SMs)
  std::vector<std::vector<cudaStream_t>> side;
  std::vector<cudaEvent_t> fork_ev;
  std::vector<std::vector<cudaEvent_t>> join_ev;
  // pipeline slices (one device listed several times): the slices' bulk copies go through ONE stream per direction
  // and device, in slice order, so that slice k computes while slice k+1 uploads and slice k-1 downloads -- on
  // separate streams the copy engines would share the link and every slice would finish its copy at the same time
  std::vector<cudaStream_t> copy_in, copy_out;  // per ctx device entry; replicas share the handles
  std::vector<bool> own_copy;
  std::vector<cudaEvent_t> in_ev, out_ev, maps_ev;
  std::shared_ptr<DevPool> pool = std::make_shared<DevPool>();
  // DCB_DEBUG_TIMING: per-launch events of the last decode (name, begin, end), printed by finish_stats
  std::vector<std::pair<std::string, std::pair<cudaEvent_t, cudaEvent_t>>> timeline;
  dcb_launch_stats stats{};
  std::vector<dcb_launch_stats> dev_stats;  // per context device entry (entry 0 unused)
  std::vector<std::pair<const void *, uint32_t>> par_streams;  // (shard, stream): Tagged streams whose bit-area length is device-known
  // plausibility limits of one buffer (dcb_set_limits): a forged point / entry count must fail its own buffer instead
  // of sizing a 25 GB arena for the whole batch
  uint64_t max_points = 0;                          // absolute cap per buffer, 0 = none
  uint64_t points_per_byte = kDefaultPointsPerByte; // n_points <= 65536 + points_per_byte * buffer_len, 0 = unchecked
  cudaEvent_t ev[10] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool ev_raw = false, ev_tag = false, ev_par = false, ev_para = false;
  uint64_t algo_raw = 0, algo_tag = 0, algo_par = 0;
  char raw_name[96] = {0};
};

struct dcb_batch {
  std::vector<BufRec> bufs;
  std::vector<Shard> shards;
  const uint8_t *host_arena = nullptr;  // dcb_index_arena: buffers live in one host arena
  uint64_t total_out = 0, total_dbg = 0, total_in = 0, total_points = 0, algo_bytes = 0;
  int n_devices = 1;
  uint64_t max_points = 0, points_per_byte = 0;  // plausibility limits (dcb_set_limits), copied from the context
  int order = DCB_ORDER_ENTRIES;
  int faces = DCB_FACES_NONE;
  bool conn_done = false;  // dcb_index_finish has run: a new order or new faces rerun it
};

namespace {

#define CUDA_TRY(x)                          \
  do {                                       \
    cudaError_t e_ = (x);                    \
    if (e_ != cudaSuccess) {                 \
      cudaGetLastError();                    \
      return e_ == cudaErrorMemoryAllocation ? DCB_ERR_OOM : DCB_ERR_CUDA; \
    }                                        \
  } while (0)

// ---- host reader for the container header (before the ATTRIBUTES payload) ----
struct HRd {
  const uint8_t *p;
  uint64_t len, pos;
  int err;
  bool need(uint64_t n) {
    if (err) return false;
    if (pos > len || len - pos < n) { err = DCB_ERR_EOF; return false; }
    return true;
  }
  uint32_t u8() { return need(1) ? p[pos++] : 0u; }
  uint32_t u16() { if (!need(2)) return 0; uint32_t v = p[pos] | (p[pos + 1] << 8); pos += 2; return v; }
  uint32_t u32() {
    if (!need(4)) return 0;
    uint32_t v = (uint32_t)p[pos] | ((uint32_t)p[pos + 1] << 8) | ((uint32_t)p[pos + 2] << 16) | ((uint32_t)p[pos + 3] << 24);
    pos += 4;
    return v;
  }
  uint64_t varint() {
    uint64_t result = 0;
    unsigned shift = 0;
    if (err) return 0;
    for (int i = 0; i < 10; ++i) {
      if (pos >= len) { err = DCB_ERR_EOF; return 0; }
      uint32_t b = p[pos++];
      result |= (uint64_t)(b & 0x7F) << shift;
      if (!(b & 0x80)) return result;
      shift += 7;
    }
    err = DCB_ERR_EOF;
    return 0;
  }
};

// Metadata/MetadataDecoder.cs:5-49 (skip only)
void skip_metadata_element(HRd &r, int depth) {
  if (depth > 64) { r.err = DCB_ERR_UNSUPPORTED; return; }
  uint64_t n = r.varint();
  for (uint64_t i = 0; i < n && !r.err; ++i) {
    uint32_t ks = r.u8();
    if (r.need(ks)) r.pos += ks;
    uint32_t vs = r.u8();
    if (r.need(vs)) r.pos += vs;
  }
  uint64_t ns = r.varint();
  for (uint64_t i = 0; i < ns && !r.err; ++i) {
    uint32_t ks = r.u8();
    if (r.need(ks)) r.pos += ks;
    skip_metadata_element(r, depth + 1);
  }
}
void skip_metadata(HRd &r) {
  uint64_t n = r.varint();
  for (uint64_t i = 0; i < n && !r.err; ++i) {
    (void)r.varint();
    skip_metadata_element(r, 0);
  }
  skip_metadata_element(r, 0);
}

// DracoDecoder.DecodeHeader + the connectivity prefix that is host business.  Fills info; returns
// the offset of the ATTRIBUTES section for geometry the library can walk on its own.
void parse_header(BufRec &b) {
  dcb_buffer_info &inf = b.info;
  memset(&inf, 0, sizeof inf);
  HRd r{b.src, b.len, 0, 0};
  if (!r.need(5)) { inf.status = DCB_ERR_EOF; return; }
  if (memcmp(b.src, "DRACO", 5) != 0) { inf.status = DCB_ERR_MAGIC; return; }
  r.pos = 5;
  inf.version_major = (int32_t)r.u8();
  inf.version_minor = (int32_t)r.u8();
  inf.geometry_type = (int32_t)r.u8();
  inf.encoder_method = (int32_t)r.u8();
  inf.flags = (int32_t)r.u16();
  if (r.err) { inf.status = r.err; return; }
  if (inf.version_major != 2 || inf.version_minor != 2) { inf.status = DCB_ERR_UNSUPPORTED; return; }
  if (inf.flags & 0x8000) skip_metadata(r);
  if (r.err) { inf.status = r.err; return; }
  if (inf.geometry_type == 0) {  // point cloud (B-1: upstream sequential container)
    if (inf.encoder_method != 0) { inf.status = DCB_ERR_UNSUPPORTED; return; }  // kd-tree: absent from the reference
    int32_t np = (int32_t)r.u32();
    if (r.err) { inf.status = r.err; return; }
    if (np < 0) { inf.status = DCB_ERR_ATTR; return; }
    inf.n_points = (uint32_t)np;
    inf.attr_section_off = r.pos;
  } else if (inf.geometry_type == 1) {
    b.conn_off = r.pos;
    if (inf.encoder_method == 1) {
      // Edgebreaker: connectivity is host work (DracoDecoder.cs:80-88 -> MeshEdgeBreakerDecoder); the
      // caller reports where ATTRIBUTES starts with dcb_set_attr_section + dcb_set_mesh_maps.
      b.is_eb = true;
      inf.needs_connectivity = 1;
    } else if (inf.encoder_method == 0) {
      // sequential mesh connectivity (MeshSequentialDecoder.cs:8-118): host work as well
      inf.needs_connectivity = 1;
    } else {
      inf.status = DCB_ERR_UNSUPPORTED;
    }
  } else {
    inf.status = DCB_ERR_UNSUPPORTED;
  }
}

// A point / entry count that the buffer's own size cannot plausibly back fails THIS buffer (DCB_ERR_ATTR) before it
// sizes any arena.  The rule is deliberately loose -- a constant attribute legitimately costs ~0 bits per point -- and
// caller-settable (dcb_set_limits).
bool implausible(const dcb_batch &b, uint64_t n_points, uint64_t len) {
  if (b.max_points && n_points > b.max_points) return true;
  if (b.points_per_byte && n_points > 65536 + b.points_per_byte * len) return true;
  return false;
}
void check_plausible(const dcb_batch &b, BufRec &r) {
  if (r.info.status == DCB_OK && implausible(b, r.info.n_points, r.len)) r.info.status = DCB_ERR_ATTR;
}

// bytes of one value (StoreTypedValues; normals: three float32)
uint64_t row_bytes(const StreamDesc &s) {
  return (s.seq_type == SEQ_NORMALS) ? 12ull : (uint64_t)dcb_dtype_len(s.data_type) * s.nc;
}

// Point order walks the faces over the corners of every attributes decoder of an Edgebreaker buffer: they must be set
// and have the corner count of each decoder (whose maps the indexer has checked are there).
bool point_faces_ok(const BufRec &b, int n_dec) {
  if (!b.pt_faces_set) return false;
  if (n_dec <= 0) return true;
  const uint64_t n_face_corners = b.pt_faces ? 3 * b.pt_n_faces : b.maps[0].n_corners;
  for (int d = 0; d < n_dec; ++d)
    if (b.maps[d].n_corners != n_face_corners) return false;
  return true;
}

// DCB_FACES_ARENA: a mesh needs faces to put in the arena -- installed by dcb_host_connectivity or (Edgebreaker)
// dcb_set_mesh_faces; the NULL form needs the corner table of attributes decoder 0
bool faces_known(const BufRec &b) {
  if (!b.pt_faces_set) return false;
  return !b.is_eb || b.pt_faces || (!b.maps.empty() && b.maps[0].set);
}

// DEC_ID + DEC_DATA: creates the StreamDescs of one buffer (appended to sh.streams) and its BufWalk.
void parse_attr_section(BufRec &b, Shard &sh, int buf_index, const dcb_batch *batch = nullptr) {
  dcb_buffer_info &inf = b.info;
  BufWalk w;
  memset(&w, 0, sizeof w);
  w.begin = b.arena_off;
  w.end = b.arena_off + b.len;
  w.stream_first = (int32_t)sh.streams.size();
  w.blocked = -1;
  w.phase = 2;
  w.geom_type = (uint8_t)inf.geometry_type;
  w.method = (uint8_t)inf.encoder_method;
  auto finish = [&](int status) {
    if (status && !inf.status) inf.status = status;
    w.status = inf.status;
    w.stream_count = (int32_t)sh.streams.size() - w.stream_first;
    inf.n_attrs = w.stream_count;
    sh.walks[b.local] = w;
  };
  if (inf.status) return finish(inf.status);
  if (inf.needs_connectivity) return finish(0);  // attributes are indexed by dcb_index_finish
  if (batch && batch->faces == DCB_FACES_ARENA && inf.geometry_type == 1 && !faces_known(b)) {
    b.pt_failed = true;
    return finish(DCB_ERR_MAPS);
  }
  HRd r{b.src, b.len, inf.attr_section_off, 0};
  const int n_dec = (int)r.u8();  // ConnectivityDecoder.cs:18
  if (r.err) return finish(r.err);
  inf.n_attr_decoders = n_dec;
  if (b.is_eb) {  // DEC_ID: MeshEdgeBreakerDecoder.cs:642-662 (att_data_id, decoder type, traversal method)
    for (int i = 0; i < n_dec; ++i) { r.u8(); r.u8(); r.u8(); }
    if (r.err) return finish(r.err);
  }
  for (int d = 0; d < n_dec; ++d) {
    uint64_t na = r.varint();
    if (r.err) return finish(r.err);
    if (na > (b.len - r.pos)) return finish(DCB_ERR_EOF);
    const size_t first = sh.streams.size();
    for (uint64_t i = 0; i < na; ++i) {
      StreamDesc s;
      memset(&s, 0, sizeof s);
      s.buf_begin = w.begin;
      s.buf_end = w.end;
      s.buf_index = buf_index;
      s.attr_index = (int32_t)(sh.streams.size() - (size_t)w.stream_first);
      s.decoder_id = (uint8_t)d;
      s.scheme = SCHEME_EMPTY;
      s.pred_method = PRED_NONE;
      s.transform = XF_NONE;
      s.att_type = (uint8_t)r.u8();
      s.data_type = (uint8_t)r.u8();
      s.nc = (uint8_t)r.u8();
      s.normalized = r.u8() != 0;
      s.unique_id = (uint32_t)r.varint();
      sh.streams.push_back(s);
      if (r.err) return finish(r.err);
      if (s.att_type >= 5 || s.data_type == 0 || s.data_type >= DT_COUNT || s.nc == 0) return finish(DCB_ERR_ATTR);
    }
    int status = 0;
    for (uint64_t i = 0; i < na && !status; ++i) {
      StreamDesc &s = sh.streams[first + i];
      s.seq_type = (uint8_t)r.u8();
      if (r.err) { status = r.err; break; }
      if (s.seq_type > 3) { status = DCB_ERR_UNSUPPORTED; break; }
      if (s.seq_type == SEQ_QUANTIZATION && s.data_type != DT_FLOAT32) status = DCB_ERR_ATTR;
      if (s.seq_type == SEQ_NORMALS && (s.data_type != DT_FLOAT32 || s.nc != 3)) status = DCB_ERR_ATTR;
      s.ncp = (s.seq_type == SEQ_NORMALS) ? 2 : s.nc;  // AttributeOctahedronTransform.cs:23-26, B-8
      if (s.nc > 4 && s.seq_type == SEQ_QUANTIZATION) status = DCB_ERR_UNSUPPORTED;
      // the fast kernels are specialised for 1..4 portable components; integer attributes with more (the reference loops
      // over any nc, SequentialIntegerAttributeDecoder.cs:144-152) take the generic wide path (wide_post_kernel)
      if (!status && s.seq_type != SEQ_GENERIC && s.seq_type != SEQ_INTEGER && s.ncp > 4) status = DCB_ERR_UNSUPPORTED;
    }
    if (status) return finish(status);
    // entry count of this decoder: LinearSequencer.cs:7-13 (B-2) / traversal observer for Edgebreaker
    uint32_t n_entries = inf.n_points;
    bool has_maps = false;
    if (b.is_eb) {
      if ((size_t)d >= b.maps.size() || !b.maps[d].set) return finish(DCB_ERR_MAPS);
      n_entries = (uint32_t)b.maps[d].n_entries;
      has_maps = true;
      if (batch && implausible(*batch, n_entries, b.len)) return finish(DCB_ERR_ATTR);
    }
    for (uint64_t i = 0; i < na; ++i) {
      StreamDesc &s = sh.streams[first + i];
      s.n_entries = n_entries;
      s.has_maps = has_maps ? 1 : 0;
      if (has_maps) {
        s.n_corners = (uint32_t)b.maps[d].n_corners;
        s.n_vertices = (uint32_t)b.maps[d].n_vertices;
      }
      s.out_bytes = row_bytes(s) * n_entries;
    }
  }
  if (b.is_eb && batch && batch->order == DCB_ORDER_POINTS && n_dec > 0) {
    if (!point_faces_ok(b, n_dec)) {
      b.pt_failed = true;
      return finish(DCB_ERR_MAPS);
    }
  }
  w.pos = b.arena_off + r.pos;
  w.stream_count = (int32_t)sh.streams.size() - w.stream_first;
  w.phase = w.stream_count > 0 ? 0 : 2;
  {  // parent of the tex-coord predictor: PointCloud.GetNamedAttributeId(Position) = the buffer's first position
     // attribute (SequentialAttributeDecoder.InitPredictionScheme :58-72)
    int32_t pos_stream = -1;
    for (int i = 0; i < w.stream_count && pos_stream < 0; ++i)
      if (sh.streams[(size_t)w.stream_first + i].att_type == 0) pos_stream = w.stream_first + i;
    for (int i = 0; i < w.stream_count; ++i) sh.streams[(size_t)w.stream_first + i].parent = pos_stream;
  }
  // host part of the payload walk (stops at the first Tagged bit area)
  if (w.stream_count > 0) walk_continue(b.src - b.arena_off, w, sh.streams.data());
  finish(w.status);
}

cudaError_t pool_alloc(const std::shared_ptr<DevPool> &pool, int device, uint64_t bytes, uint8_t **out, uint64_t *cap) {
  *out = nullptr;
  *cap = 0;
  if (bytes == 0) return cudaSuccess;
  std::unique_lock<std::mutex> lk_;
  if (pool) lk_ = std::unique_lock<std::mutex>(pool->mu);
  if (pool && bytes >= kPoolMin) {
    int best = -1;
    for (size_t i = 0; i < pool->free_blocks.size(); ++i) {
      const PoolBlock &k = pool->free_blocks[i];
      if (k.device != device || k.bytes < bytes || k.bytes > 2 * bytes) continue;
      if (best < 0 || k.bytes < pool->free_blocks[best].bytes) best = (int)i;
    }
    if (best >= 0) {
      *out = (uint8_t *)pool->free_blocks[best].p;
      *cap = pool->free_blocks[best].bytes;
      pool->cached -= *cap;
      pool->free_blocks.erase(pool->free_blocks.begin() + best);
      return cudaSuccess;
    }
  }
  const uint64_t want = bytes >= (1ull << 20) ? align_up(bytes, 2ull << 20) : align_up(bytes, 512);
  cudaError_t e = cudaMalloc(out, want);
  if (e != cudaSuccess && pool && !pool->free_blocks.empty()) {  // out of memory with a warm cache: drop it and retry
    cudaGetLastError();
    for (PoolBlock &k : pool->free_blocks) { cudaSetDevice(k.device); cudaFree(k.p); }
    pool->free_blocks.clear();
    pool->cached = 0;
    cudaSetDevice(device);
    e = cudaMalloc(out, want);
  }
  if (e == cudaSuccess) *cap = want;
  return e;
}

void pool_free(const std::shared_ptr<DevPool> &pool, int device, void *p, uint64_t cap) {
  if (!p) return;
  std::unique_lock<std::mutex> lk_;
  if (pool) lk_ = std::unique_lock<std::mutex>(pool->mu);
  if (pool && cap >= kPoolMin && pool->cached + cap <= kPoolCap) {
    pool->free_blocks.push_back({p, cap, device});
    pool->cached += cap;
    return;
  }
  cudaFree(p);
}

void pool_trim(const std::shared_ptr<DevPool> &pool) {
  if (!pool) return;
  std::unique_lock<std::mutex> lk_;
  if (pool) lk_ = std::unique_lock<std::mutex>(pool->mu);
  for (PoolBlock &k : pool->free_blocks) { cudaSetDevice(k.device); cudaFree(k.p); }
  for (PoolBlock &k : pool->free_pinned) cudaFreeHost(k.p);
  pool->free_blocks.clear();
  pool->free_pinned.clear();
  pool->cached = 0;
}

cudaError_t pinned_alloc(const std::shared_ptr<DevPool> &pool, uint64_t bytes, uint8_t **out, uint64_t *cap) {
  std::unique_lock<std::mutex> lk_;
  if (pool) lk_ = std::unique_lock<std::mutex>(pool->mu);
  if (pool)
    for (size_t i = 0; i < pool->free_pinned.size(); ++i) {
      const PoolBlock k = pool->free_pinned[i];
      if (k.bytes >= bytes && k.bytes <= 2 * bytes + 4096) {
        *out = (uint8_t *)k.p;
        *cap = k.bytes;
        pool->free_pinned.erase(pool->free_pinned.begin() + i);
        return cudaSuccess;
      }
    }
  *cap = align_up(bytes, 4096);
  return cudaMallocHost(out, *cap);
}

void pinned_free(const std::shared_ptr<DevPool> &pool, void *p, uint64_t cap) {
  if (!p) return;
  std::unique_lock<std::mutex> lk_;
  if (pool) lk_ = std::unique_lock<std::mutex>(pool->mu);
  if (pool && pool->cached <= kPoolCap && pool->free_pinned.size() < 64) {
    pool->free_pinned.push_back({p, cap, -1});
    return;
  }
  cudaFreeHost(p);
}

void pinned_free(const std::shared_ptr<DevPool> &pool, void *p, uint64_t cap);
void free_shard_device(Shard &sh) {
  if (sh.h_desc) {
    pinned_free(sh.pool, sh.h_desc, sh.cap_hdesc);
    sh.h_desc = nullptr;
    sh.desc_pending = false;
  }
  if (!sh.d_in && !sh.d_streams && !sh.h_stage && !sh.d_out && !sh.h_maps) return;
  cudaSetDevice(sh.device);
  pool_free(sh.pool, sh.device, sh.d_in, sh.cap_in);
  if (sh.own_out) pool_free(sh.pool, sh.device, sh.d_out, sh.cap_out);
  cudaFree(sh.d_dbg);
  pool_free(sh.pool, sh.device, sh.d_aux, sh.cap_aux);
  cudaFree(sh.d_tab);
  pool_free(sh.pool, sh.device, sh.d_maps, sh.cap_maps);
  pool_free(sh.pool, sh.device, sh.d_streams, sh.cap_streams);
  pool_free(sh.pool, sh.device, sh.d_walks, sh.cap_walks);
  pool_free(sh.pool, sh.device, sh.d_order, sh.cap_order);
  pool_free(sh.pool, sh.device, sh.d_pts, sh.cap_pts);
  sh.d_pts = nullptr;
  pool_free(sh.pool, sh.device, sh.d_faces, sh.cap_faces);
  sh.d_faces = nullptr;
  if (sh.h_fstatus) pinned_free(sh.pool, sh.h_fstatus, sh.cap_hfstatus);
  sh.h_fstatus = nullptr;
  if (sh.h_stage) pinned_free(sh.pool, sh.h_stage, sh.cap_stage);
  if (sh.h_maps) pinned_free(sh.pool, sh.h_maps, sh.cap_hmaps);
  sh.h_maps = nullptr;
  sh.d_in = sh.d_out = sh.d_dbg = sh.d_aux = sh.d_tab = sh.d_maps = nullptr;
  sh.d_streams = nullptr;
  sh.d_walks = nullptr;
  sh.d_order = nullptr;
  sh.h_stage = nullptr;
  sh.uploaded = false;
}

// Lay out outputs / scratch of a shard once its streams exist.
void layout_shard(Shard &sh) {
  uint64_t out = 0, dbg = 0, aux = 0;
  for (size_t bi = 0; bi < sh.walks.size(); ++bi) {
    const BufWalk &w = sh.walks[bi];
    bool any_unready = false;
    for (int i = 0; i < w.stream_count; ++i) {
      const StreamDesc &s = sh.streams[w.stream_first + i];
      if (s.state < ST_READY || s.scheme == SCHEME_TAGGED) any_unready = true;
    }
    for (int i = 0; i < w.stream_count; ++i) {
      StreamDesc &s = sh.streams[w.stream_first + i];
      if (w.status) {  // a buffer that failed while indexing reserves no output, debug or scratch space
        s.out_off = out;
        s.dbg_off = dbg;
        s.out_bytes = 0;
        continue;
      }
      s.out_off = out;
      out = align_up(out + s.out_bytes, 128);
      const uint64_t nv = (uint64_t)s.n_entries * (s.ncp ? s.ncp : s.nc);
      s.dbg_off = dbg;
      dbg = align_up(dbg + nv * 4, 16);
      if (s.seq_type != SEQ_GENERIC &&
          (s.scheme == SCHEME_TAGGED || s.scheme == SCHEME_UNCOMPRESSED || (any_unready && s.state < ST_READY))) {
        // tags u8[n] | bit offset per chunk u64[nch + 1] | look-back state words per chunk u64[nch][4]
        const uint64_t nch = (s.n_entries + DCB_TAG_CHUNK - 1) / DCB_TAG_CHUNK;
        s.tag_off = aux;
        aux = align_up(aux + align_up(s.n_entries, 16) + 8ull * (nch + 1) + 32ull * nch, 16);
      }
      if (s.seq_type != SEQ_GENERIC && s.has_maps && (s.recon == RECON_PARA_WRAP || s.state < ST_READY)) {
        // corrections int32[nv] | quantized ints int32[nv] | parallelogram: deps int32[3 n]; tex coords (two components):
        // TexRec[n] (32 bytes each) + orientation flags u8[<= 2n + 1]
        // constrained multi-parallelogram: deps int32[12 n] | count u8[n] | crease flags u8[10 n] (CmpScratch, dcb_cmp.cu).
        // A stream the host walk has not reached yet (behind a Tagged bit area) may turn out to be any of them.
        s.aux_off = aux;
        const uint64_t n = s.n_entries;
        const uint64_t t_para = 12ull * n, t_tex = 34ull * n + 16ull, t_cmp = 59ull * n + 48ull;
        uint64_t tail;
        if (s.state == ST_UNPARSED) tail = std::max(t_cmp, s.ncp == 2 ? t_tex : t_para);
        else if (s.pred_method == PRED_CONSTRAINED_MULTI) tail = t_cmp;
        else tail = s.ncp == 2 ? t_tex : t_para;
        aux = align_up(aux + 2ull * nv * 4 + tail, 16);
      } else if (s.seq_type == SEQ_NORMALS) {
        s.aux_off = aux;  // quantized octahedral (s, t) pairs between the serial kernels and oct_unit_kernel
        // (+ geometric normal, a mesh predictor: flip bits u8[n] behind the pairs)
        aux = align_up(aux + (s.has_maps ? 9ull : 8ull) * s.n_entries + 16ull, 16);
      } else if (s.seq_type == SEQ_INTEGER && s.ncp > 4) {
        s.aux_off = aux;  // wide attributes: zig-zag decoded symbols of a Raw source, int32[n * nc]
        aux = align_up(aux + 4ull * nv, 16);
      }
    }
  }
  sh.out_bytes = out;
  sh.dbg_bytes = dbg;
  sh.aux_bytes = aux;
}

int make_batch(dcb_ctx *ctx, const uint8_t *arena, const uint8_t *const *ptrs, const uint64_t *offs,
               const uint64_t *lens, int n_bufs, dcb_batch **out) {
  if (!out || n_bufs < 0 || (n_bufs > 0 && !lens) || (n_bufs > 0 && !arena && !ptrs)) return DCB_ERR_ARG;
  std::unique_ptr<dcb_batch> owner(new (std::nothrow) dcb_batch());
  dcb_batch *b = owner.get();
  if (!b) return DCB_ERR_OOM;
  b->max_points = ctx ? ctx->max_points : 0;
  b->points_per_byte = ctx ? ctx->points_per_byte : kDefaultPointsPerByte;
  b->n_devices = ctx ? (int)ctx->devices.size() : 1;
  b->host_arena = arena;
  b->bufs.resize((size_t)n_bufs);
  b->shards.resize((size_t)b->n_devices);
  for (int d = 0; d < b->n_devices; ++d) b->shards[d].device = ctx ? ctx->devices[d] : 0;
  bool aligned = arena != nullptr;
  for (int k = 0; k < n_bufs; ++k) {
    BufRec &r = b->bufs[k];
    r.src = arena ? arena + offs[k] : ptrs[k];
    r.len = lens[k];
    if (arena && (offs[k] & 15)) aligned = false;
    if (!r.src && r.len) return DCB_ERR_ARG;
  }
  // shard by buffer (SURVEY 8e); no collective.  Distinct devices: longest-processing-time-first on compressed bytes.
  // The same device listed K times (dcb_create): K pipeline slices -- contiguous runs of buffers with equal bytes, so
  // that each slice uploads one arena range and H2D / kernels / D2H of neighbouring slices overlap.
  std::vector<int> idx((size_t)n_bufs);
  for (int k = 0; k < n_bufs; ++k) idx[k] = k;
  std::vector<uint64_t> load((size_t)b->n_devices, 0);
  bool replicas = b->n_devices > 1;
  for (int d = 1; d < b->n_devices; ++d) replicas = replicas && b->shards[d].device == b->shards[0].device;
  for (int d = 0; d < b->n_devices; ++d) {
    int share = 0;
    for (int e = 0; e < b->n_devices; ++e) share += b->shards[e].device == b->shards[d].device;
    b->shards[d].share = share;
  }
  if (replicas) {
    uint64_t total = 0, run = 0;
    for (int k = 0; k < n_bufs; ++k) total += b->bufs[k].len + 64;
    for (int k = 0; k < n_bufs; ++k) {
      b->bufs[k].shard = (int)std::min<uint64_t>((uint64_t)b->n_devices - 1, run * (uint64_t)b->n_devices / std::max<uint64_t>(total, 1));
      run += b->bufs[k].len + 64;
    }
  } else if (b->n_devices > 1) {
    std::stable_sort(idx.begin(), idx.end(), [&](int x, int y) { return b->bufs[x].len > b->bufs[y].len; });
    for (int k : idx) {
      int best = 0;
      for (int d = 1; d < b->n_devices; ++d)
        if (load[d] < load[best]) best = d;
      b->bufs[k].shard = best;
      load[best] += b->bufs[k].len + 64;
    }
  }
  for (int k = 0; k < n_bufs; ++k) {
    Shard &sh = b->shards[b->bufs[k].shard];
    b->bufs[k].local = (int)sh.bufs.size();
    sh.bufs.push_back(k);
  }
  for (Shard &sh : b->shards) {
    sh.direct = aligned && !sh.bufs.empty() && (b->n_devices == 1 || replicas);
    if (sh.direct) {
      uint64_t lo = ~0ull, hi = 0;
      for (int k : sh.bufs) {
        lo = std::min(lo, offs[k]);
        hi = std::max(hi, offs[k] + lens[k]);
      }
      // a slice must not drag foreign bytes along: its range may only hold its own buffers (arena in buffer order)
      uint64_t own = 0;
      for (int k : sh.bufs) own += lens[k];
      if (b->n_devices > 1 && hi - lo > own + 64ull * sh.bufs.size()) sh.direct = false;
      if (sh.direct) {
        sh.direct_lo = lo;
        sh.direct_hi = hi;
        for (int k : sh.bufs) b->bufs[k].arena_off = kFrontPad + (offs[k] - lo);
        sh.in_bytes = kFrontPad + (hi - lo) + kBackPad;
      }
    }
    if (!sh.direct) {
      uint64_t pos = kFrontPad;
      for (int k : sh.bufs) {
        b->bufs[k].arena_off = pos;
        pos = align_up(pos + b->bufs[k].len, 16);
      }
      sh.in_bytes = pos + kBackPad;
    }
  }
  for (Shard &sh : b->shards) sh.walks.resize(sh.bufs.size());
  // header + attribute indexing: a shard's buffers in order (the shard's stream list is append-only), shards in
  // parallel when there are several -- nothing is shared between them
  std::atomic<bool> index_oom{false};
  auto index_shard = [&](Shard &sh) {
    try {
      for (int k : sh.bufs) {
        BufRec &r = b->bufs[k];
        parse_header(r);
        r.info.device = r.shard;
        check_plausible(*b, r);
        parse_attr_section(r, sh, k, b);
      }
    } catch (...) {  // std::bad_alloc inside a worker thread must not reach std::terminate
      index_oom = true;
    }
  };
  if (b->n_devices > 1 && n_bufs >= 16) {
    std::vector<std::thread> th;
    for (Shard &sh : b->shards) th.emplace_back(index_shard, std::ref(sh));
    for (std::thread &t : th) t.join();
  } else {
    for (Shard &sh : b->shards) index_shard(sh);
  }
  if (index_oom) return DCB_ERR_OOM;
  *out = owner.release();
  return DCB_OK;
}

// The caller's view of the output arena.  Entry order: the kernels' layout.  Point order: a shard holding an indexed
// Edgebreaker buffer stages the kernels' entry-order layout (stage_bytes) and lays the output arena out again with
// n_points rows for the attributes of its Edgebreaker buffers; every attribute keeps its place in (buffer, attribute)
// order on a 128-byte boundary.
void layout_points(const dcb_batch *b, Shard &sh) {
  const size_t n = sh.streams.size();
  sh.fin_off.resize(n);
  sh.fin_bytes.resize(n);
  sh.pts = false;
  sh.stage_bytes = 0;
  if (b->order == DCB_ORDER_POINTS)
    for (size_t bi = 0; bi < sh.walks.size(); ++bi)
      sh.pts = sh.pts || (b->bufs[sh.bufs[bi]].is_eb && sh.walks[bi].status == DCB_OK && sh.walks[bi].stream_count > 0);
  if (!sh.pts) {
    for (size_t i = 0; i < n; ++i) {
      sh.fin_off[i] = sh.streams[i].out_off;
      sh.fin_bytes[i] = sh.streams[i].out_bytes;
    }
    return;
  }
  sh.stage_bytes = sh.out_bytes;
  uint64_t out = 0;
  for (size_t bi = 0; bi < sh.walks.size(); ++bi) {
    const BufWalk &w = sh.walks[bi];
    const BufRec &r = b->bufs[sh.bufs[bi]];
    for (int i = 0; i < w.stream_count; ++i) {
      const size_t si = (size_t)w.stream_first + i;
      const StreamDesc &s = sh.streams[si];
      const uint64_t rows = r.is_eb ? r.info.n_points : s.n_entries;
      sh.fin_off[si] = out;
      sh.fin_bytes[si] = w.status ? 0 : rows * row_bytes(s);
      out = align_up(out + sh.fin_bytes[si], 128);
    }
  }
  sh.out_bytes = out;
}

// DCB_FACES_ARENA: behind the attributes of a shard, a faces region per mesh buffer that is ok, in buffer order, each on a
// 128-byte boundary
// A sequential mesh whose Raw index differences the GPU decodes gets one more Raw rANS stream (one component, no zig-zag:
// the value map holds the raw symbol; RECON_PARA_WRAP routes the symbols to the int32 scratch as for mesh corrections),
// located by the walker code the attribute streams use, with scratch and debug space of its own.
void add_index_stream(BufRec &r, int k, Shard &sh) {
  StreamDesc s;
  memset(&s, 0, sizeof s);
  s.buf_begin = r.arena_off;
  s.buf_end = r.arena_off + r.len;
  s.buf_index = k;
  s.attr_index = -1;
  s.parent = -1;
  s.n_entries = (uint32_t)r.seq_loc.n_idx;
  s.nc = s.ncp = 1;
  s.data_type = DT_INT32;
  s.seq_type = SEQ_INTEGER;
  s.pred_method = PRED_NONE;
  s.transform = XF_NONE;
  s.scheme = SCHEME_RAW;
  s.compressed = 1;
  s.zigzag = 0;
  s.recon = RECON_PARA_WRAP;
  s.store = STORE_NARROW;
  s.max_bit_length = (uint8_t)r.seq_loc.mbl;
  s.prec_bits = (uint8_t)dcb_rans_precision(r.seq_loc.mbl);
  WalkRd wr{r.src - r.arena_off, r.arena_off + r.len, r.arena_off + r.seq_loc.off, 0};
  s.table_off = wr.pos;
  int e = walk_rans_table(wr, s.prec_bits, s.num_symbols, s.n_active, s.dense_prefix, s.narrow_blk, s.rec_need);
  if (!e) e = walk_rans_payload(wr, s.prec_bits, s.payload_off, s.payload_len);
  s.status = e;  // the host checked this stream already (dcb_host_sequential): cannot fail
  s.state = ST_READY;
  s.aux_off = align_up(sh.aux_bytes, 16);
  sh.aux_bytes = align_up(s.aux_off + 4ull * s.n_entries, 16);
  s.dbg_off = sh.dbg_bytes;
  sh.dbg_bytes = align_up(s.dbg_off + 4ull * s.n_entries, 16);
  sh.streams.push_back(s);
}

void layout_faces(dcb_batch *b, Shard &sh) {
  uint64_t out = sh.out_bytes;
  if (sh.idx_first != ~0u && sh.idx_first <= sh.streams.size()) sh.streams.resize(sh.idx_first);
  sh.idx_first = (uint32_t)sh.streams.size();
  for (int k : sh.bufs) {
    BufRec &r = b->bufs[k];
    r.face_src = 0;
    r.idx_job = -1;
    r.n_faces = r.face_off = 0;
    if (b->faces != DCB_FACES_ARENA || r.info.geometry_type != 1 || r.info.needs_connectivity || r.info.status != DCB_OK)
      continue;
    if (r.is_eb) {
      if (!r.pt_faces && (r.maps.empty() || !r.maps[0].set)) continue;  // no faces (failed at indexing; see faces_known)
      r.n_faces = r.pt_faces ? r.pt_n_faces : r.maps[0].n_corners / 3;
      r.face_src = 1;
    } else if (r.seq_loc.located) {
      if (r.seq_loc.width < 0 && r.seq_loc.n_idx) add_index_stream(r, k, sh);
      r.n_faces = r.seq_loc.n_idx / 3;
      r.face_src = 2;
    } else {
      r.n_faces = r.pt_n_faces;
      r.face_src = 1;
    }
    r.face_off = align_up(out, 128);
    out = r.face_off + 12 * r.n_faces;
  }
  sh.out_bytes = out;
}

void finalize_layout(dcb_batch *b) {
  uint64_t out_base = 0, dbg_base = 0;
  b->total_in = 0;
  b->total_points = 0;
  b->algo_bytes = 0;
  for (Shard &sh : b->shards) {
    layout_shard(sh);
    layout_points(b, sh);
    layout_faces(b, sh);  // may append index streams: before streams0
    sh.out_base = out_base;
    sh.dbg_base = dbg_base;
    out_base += align_up(sh.out_bytes, 128);
    dbg_base += align_up(sh.dbg_bytes, 128);
    sh.streams0 = sh.streams;
    sh.walks0 = sh.walks;
    sh.dirty = true;
  }
  b->total_out = out_base;
  b->total_dbg = dbg_base;
  for (const BufRec &r : b->bufs) {
    b->total_in += r.len;
    if (r.info.status == DCB_OK && !r.info.needs_connectivity) {
      b->total_points += r.info.n_points;
      b->algo_bytes += r.len;
      const Shard &sh = b->shards[r.shard];
      const BufWalk &w = sh.walks[r.local];
      for (int i = 0; i < w.stream_count; ++i) b->algo_bytes += sh.streams[w.stream_first + i].out_bytes;
      for (const MeshMapsHost &m : r.maps)
        if (m.set) b->algo_bytes += m.bytes();
      b->algo_bytes += 12 * r.n_faces;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// launch planning
// ---------------------------------------------------------------------------------------------
uint32_t ceil_log2(uint32_t v) {
  uint32_t l = 0;
  while ((1ull << l) < v) ++l;
  return l;
}

struct RawKey {
  int ncp, wide, compact, prec, size_class, zig, mode;
  bool operator<(const RawKey &o) const {
    return std::tie(ncp, wide, compact, prec, size_class, zig, mode) <
           std::tie(o.ncp, o.wide, o.compact, o.prec, o.size_class, o.zig, o.mode);
  }
};

uint32_t ent_bytes_for(const Group &g) {
  const uint32_t sz = g.wide ? 4u : 2u;
  return (uint32_t)align_up((uint64_t)(g.entries + 2u) * sz + (g.compact ? (uint64_t)g.exc * sz : 0ull), 16);
}
uint32_t lut_bytes_for(const Group &g, uint32_t k) { return ((1u << g.prec_bits) >> k) * (g.wide ? 4u : 2u); }
uint32_t lane_bytes_for(const Group &g, uint32_t k) { return lut_bytes_for(g, k) + ent_bytes_for(g) + DCB_RING_BYTES; }

// Choose LUT granularity, lanes per warp-CTA and the table home for every rANS group of a shard so
// that as many streams as possible are resident at once: the chains are serial, so the batch time
// is (waves) x (longest chain) and a second wave doubles it.
// `share`: shards decoding on the same device at the same time (pipeline slices); each plans for its part of an SM
// `corun`: bytes of every SM left free for the CTAs of kernels that run NEXT TO the rANS kernels (oct_chain, oct_unit on
// a side stream): a CTA needs its 1 KB system reservation even when it declares no shared memory, so an SM whose
// shared memory the rANS CTAs fill to the brim holds nothing else.
void plan_rans_groups(std::vector<Group *> &gs, uint32_t num_sms, uint32_t share = 1, uint32_t corun = 0) {
  share = std::max(1u, share);
  const uint32_t sm_bytes = (kSmemPerSM - corun) / share;
  const uint32_t budget = sm_bytes - std::min(sm_bytes / 2, std::max(10 * kSmemPerCtaReserve / share, 2 * kSmemPerCtaReserve + 512));
  std::vector<uint32_t> per_sm(gs.size()), kcap(gs.size());
  for (size_t i = 0; i < gs.size(); ++i) {
    Group &g = *gs[i];
    per_sm[i] = std::min<uint32_t>(1024u, (uint32_t)((g.order.size() + num_sms - 1) / num_sms));
    const uint32_t le = ceil_log2(std::max(2u, g.entries));
    const uint32_t kfloor = g.wide ? 2u : 1u;
    // finest LUT: ~4 buckets per table entry; coarsest: ~1 bucket per 4 entries (>= 16 buckets)
    uint32_t kmin = g.prec_bits > le + 2 ? g.prec_bits - le - 2 : 0;
    kmin = std::max(kmin, kfloor);
    kcap[i] = std::max(kmin, std::min<uint32_t>(g.prec_bits - 4, g.prec_bits > le ? g.prec_bits - le + 2 : 2));
    // compact u16 tables decode through the two-region byte LUT; the uniform LUT is only their fallback, keep it
    // small (2^prec / 16 bytes: also the capacity of the byte LUT's wide region) and spend the memory on region B
    if (!g.wide && g.compact) kmin = std::max(kmin, std::min<uint32_t>(5u, g.prec_bits - 4));
    kcap[i] = std::max(kcap[i], kmin);
    g.lut_shift = kmin;
  }
  auto total_for = [&]() {
    uint64_t total = 0;
    for (size_t i = 0; i < gs.size(); ++i) total += (uint64_t)per_sm[i] * lane_bytes_for(*gs[i], gs[i]->lut_shift);
    return total;
  };
  for (;;) {
    if (total_for() <= budget) break;
    int best = -1;
    uint64_t best_share = 0;
    for (size_t i = 0; i < gs.size(); ++i) {
      Group &g = *gs[i];
      if (g.lut_shift >= kcap[i]) continue;
      const uint64_t share = (uint64_t)per_sm[i] * lut_bytes_for(g, g.lut_shift);
      if (share > best_share) { best_share = share; best = (int)i; }
    }
    if (best < 0) break;
    gs[best]->lut_shift++;
  }
  // share of the SM each group may use when not everything fits: proportional to its demand
  const uint64_t total = total_for();
  for (size_t i = 0; i < gs.size(); ++i) {
    Group &g = *gs[i];
    g.ent_bytes = ent_bytes_for(g);
    g.lut_bytes = lut_bytes_for(g, g.lut_shift);
    const uint32_t lane_bytes = lane_bytes_for(g, g.lut_shift);
    g.table_global = lane_bytes > 40 * 1024;
    if (g.table_global) {
      // tables in HBM/L2 (u32 entries): LUT ~ 2 buckets per entry, any size
      g.wide = true;
      const uint32_t le = ceil_log2(std::max(2u, g.entries));
      g.lut_shift = std::max<uint32_t>(2u, g.prec_bits > le + 1 ? g.prec_bits - le - 1 : 0);
      g.ent_bytes = ent_bytes_for(g);
      g.lut_bytes = lut_bytes_for(g, g.lut_shift);
      g.lanes = 32;
      continue;
    }
    uint32_t want = per_sm[i];
    if (total > budget) {
      const uint64_t my = (uint64_t)budget * ((uint64_t)per_sm[i] * lane_bytes) / total;
      want = std::max<uint32_t>(1u, (uint32_t)(my / lane_bytes));
    }
    g.pairs = 0;
    // what the group's tables need of the two-region LUT's narrow region: it covers the slots from the first entry
    // narrower than 2^k on, for the k whose wide region still fits the LUT
    auto lutb_need = [&]() -> uint32_t {
      uint32_t need = 0xFFFFFFFFu;
      if (!g.nb_any) return need;
      const uint32_t prec = 1u << g.prec_bits;
      for (uint32_t k = 1; k <= 7; ++k) {
        if (k + 7 > g.prec_bits) continue;
        const uint32_t t_max = std::min(prec, g.nb_max[k] << 7), t_min = std::min(prec, g.nb_min[k] << 7);
        if ((t_max >> k) > g.lut_bytes) continue;
        need = std::min(need, (prec - t_min) >> 1);
      }
      return need == 0xFFFFFFFFu ? need : std::max<uint32_t>(16u, (uint32_t)align_up(need, 16));
    };
    g.direct = 0;
    const uint32_t ksym = g.tag ? 16u : 4u * (uint32_t)g.ncp;
    const uint64_t sm_cap = (uint64_t)sm_bytes + 1024 / share;
    auto pc_cta_bytes = [&](uint32_t pairs, uint32_t lanes, uint32_t lut, uint32_t lutb, uint32_t direct) -> uint64_t {
      RansLaunch L{};
      L.lanes_per_warp = lanes;
      L.lut_bytes = lut;
      L.lutb_bytes = lutb;
      L.ent_bytes = g.ent_bytes;
      L.prec_bits = g.prec_bits;
      L.pairs = pairs;
      L.direct = direct;
      return (uint64_t)dcb_rans_pc_smem_bytes(L, ksym) + kSmemPerCtaReserve;
    };
    // ---- few streams per SM: direct slot LUT + chain / consumer warp pairs (dcb_rans_pc.cu) ----
    // The batch time of a handful of long streams is chain latency and nothing else: one dependent shared-memory
    // access per symbol (slot -> {freq, offset}, 6 bytes per slot) instead of two, and a chain warp that carries
    // nothing but the chain; its consumer warp sits on another sub-partition (two pairs per CTA: warps 0,1 are
    // chain warps, 2,3 their consumers).  Taken whenever every stream of the group is resident that way.
    if (!g.wide && g.prec_bits <= 15 && !env_flags().no_direct && !g.no_direct && per_sm[i] <= 64 && want == per_sm[i]) {
      const uint32_t pairs = std::min<uint32_t>(2u, want), lanes = (want + pairs - 1) / pairs;
      const uint32_t dlut = 6u << g.prec_bits;
      if ((uint64_t)lanes * g.ent_bytes <= 65535 && pc_cta_bytes(pairs, lanes, dlut, 0, 1) <= sm_cap) {
        g.direct = 1;
        g.pairs = pairs;
        g.lanes = lanes;
        g.lut_bytes = dlut;
        g.lutb_bytes = 0;
        continue;
      }
    }
    // ---- bucket-record tables (dcb_rans_rec.cu): one dependent shared-memory access per symbol, warp pairs, one CTA of
    // up to four pairs per SM.  Taken whenever every stream of the group has the table shape and is resident that way.
    g.rec_ka = 0;
    g.split = 0;
    if (!g.wide && g.prec_bits <= 15 && g.nb_any && !env_flags().no_rec && !env_flags().rans_pc && !g.force_single_warp && want == per_sm[i] && want <= 128) {
      const bool split = env_flags().split && share == 1;
      const uint32_t pairs = std::min<uint32_t>(split ? 3u : std::max<uint32_t>(1u, 4u / share), want), lanes = (want + pairs - 1) / pairs;
      uint32_t best_j = 4, best_bytes = 0xFFFFFFFFu;
      for (uint32_t j = 0; j < 4; ++j) {
        if (g.rec_max[j] >= 0xFFFFu || DCB_REC_KA0 + j >= g.prec_bits) continue;
        if (env_flags().rec_ka > 0 && (uint32_t)env_flags().rec_ka != DCB_REC_KA0 + j) continue;
        const uint32_t bytes = 8u * g.rec_max[j] + (uint32_t)align_up(2ull * g.exc_all, 8);
        if (bytes < best_bytes) { best_bytes = bytes; best_j = j; }
      }
      if (best_j < 4 && lanes <= 32) {
        RansLaunch L{};
        L.lanes_per_warp = lanes;
        L.prec_bits = g.prec_bits;
        L.pairs = pairs;
        L.rec_ka = DCB_REC_KA0 + best_j;
        L.rec_bytes = best_bytes;
        if ((uint64_t)dcb_rans_rec_smem_bytes(L, ksym) + kSmemPerCtaReserve <= sm_cap) {
          g.rec_ka = L.rec_ka;
          g.rec_bytes = best_bytes;
          g.split = split ? 1u : 0u;
          g.pairs = pairs;
          g.lanes = lanes;
          g.lutb_bytes = 0;
          continue;
        }
      }
    }
    if (!g.wide && env_flags().rans_pc && !g.force_single_warp) {
      // ---- chain / consumer warp pairs with the two-level tables (experiment: measured slower than one warp per
      // sub-partition when the SM is full of streams -- the two warps of a pair compete for the same issue port) ----
      const uint32_t target = std::max<uint32_t>(1u, 4u / share);
      const uint32_t lutb_min = g.compact ? 16u : 0u;
      uint32_t pairs = 1, lanes = 1, ctas = 1;
      if (env_flags().split && share == 1 && (want + 2) / 3 <= 32) {
        // split layout: one CTA per SM, three chain warps with a sub-partition each, their consumers on the fourth
        const uint32_t lutb_min0 = g.compact ? 16u : 0u;
        const uint32_t p3 = std::min<uint32_t>(3u, want), l3 = (want + p3 - 1) / p3;
        if ((uint64_t)l3 * g.ent_bytes <= 65535 && pc_cta_bytes(p3, l3, g.lut_bytes, lutb_min0, 0) <= sm_cap) {
          g.split = 1;
          g.lanes = l3;
          g.pairs = p3;
          g.lutb_bytes = 0;
          if (g.compact) {
            const uint64_t base = pc_cta_bytes(p3, l3, g.lut_bytes, lutb_min0, 0);
            const uint64_t spare = sm_cap > base ? (sm_cap - base) / ((uint64_t)p3 * (l3 + 1)) : 0;
            g.lutb_bytes = (uint32_t)std::min<uint64_t>((1u << g.prec_bits) >> 1, lutb_min0 + spare / 16 * 16);
            const uint32_t need = lutb_need();
            if (need != 0xFFFFFFFFu && !env_flags().lutb_full) g.lutb_bytes = std::min(g.lutb_bytes, need);
          }
          continue;
        }
      }
      for (;; --want) {
        uint32_t nw = std::max<uint32_t>((want + 31) / 32, std::min<uint32_t>(target, want));
        while ((uint64_t)((want + nw - 1) / nw) * g.ent_bytes > 65535) ++nw;  // 16-bit entry offsets inside a pair
        ctas = (nw + 3) / 4;
        pairs = (nw + ctas - 1) / ctas;
        lanes = (want + pairs * ctas - 1) / (pairs * ctas);
        if (ctas * pc_cta_bytes(pairs, lanes, g.lut_bytes, lutb_min, 0) <= sm_cap || want <= 1) break;
      }
      g.lanes = lanes;
      g.pairs = pairs;
      g.lutb_bytes = 0;
      if (g.compact) {
        const uint64_t base = ctas * pc_cta_bytes(pairs, lanes, g.lut_bytes, lutb_min, 0);
        const uint64_t spare = sm_cap > base ? (sm_cap - base) / ((uint64_t)ctas * pairs * (lanes + 1)) : 0;
        g.lutb_bytes = (uint32_t)std::min<uint64_t>((1u << g.prec_bits) >> 1, lutb_min + spare / 16 * 16);
        const uint32_t need = lutb_need();
        if (need != 0xFFFFFFFFu && !env_flags().lutb_full) g.lutb_bytes = std::min(g.lutb_bytes, need);
      }
      continue;
    }
    // ---- one warp per CTA (dcb_kernels.cu): spread the streams of an SM over its four sub-partitions ----
    const uint32_t ctas = std::max<uint32_t>((want + 31) / 32, std::min<uint32_t>(std::max<uint32_t>(1u, 4u / share), want));
    g.lanes = std::max<uint32_t>(1u, std::min<uint32_t>(32u, (want + ctas - 1) / ctas));
    // a CTA must fit an SM (with its alignment slack) and, for u16 tables, address its entries with 16 bits
    while (g.lanes > 1 && ((uint64_t)g.lanes * lane_bytes + g.lut_bytes + 256 > kSmemPerSM - kSmemPerCtaReserve ||
                           (!g.wide && (uint64_t)g.lanes * g.ent_bytes > 65535)))
      --g.lanes;
    // two-region LUT (compact u16 tables): give its narrow region whatever shared memory is left per lane, up
    // to one byte per two slots
    g.lutb_bytes = 0;
    if (!g.wide && g.compact) {
      const uint32_t ctas_per_sm = std::max<uint32_t>(1u, (want + g.lanes - 1) / g.lanes);
      const uint32_t blk = std::max(16u, ((1u << g.prec_bits) >> 7) << 2);
      const uint64_t cta_raw = (sm_bytes + 1024 / share) / ctas_per_sm;
      const uint64_t cta_fixed = (uint64_t)kSmemPerCtaReserve + g.lut_bytes + blk + 256;
      const uint64_t cta_budget = cta_raw > cta_fixed ? cta_raw - cta_fixed : 0;
      const uint64_t used = (uint64_t)g.lanes * (lane_bytes + blk);
      if (cta_budget > used) {
        const uint64_t spare = (cta_budget - used) / g.lanes;
        g.lutb_bytes = (uint32_t)std::min<uint64_t>((1u << g.prec_bits) >> 1, spare / 16 * 16);
      }
      // ... but no more than the group's tables need: region B covers the slots from the first entry narrower than
      // 2^k on, for the k whose wide region still fits the LUT.  What is not taken stays free for the CTAs of the
      // batch's other groups, which then run next to this one instead of behind it.
      if (g.lutb_bytes) {
        const uint32_t need = lutb_need();
        if (need != 0xFFFFFFFFu && !env_flags().lutb_full) g.lutb_bytes = std::min<uint32_t>(g.lutb_bytes, need);
      }
    }
  }
}

int ensure_order(Shard &sh, uint64_t n) {
  if (n <= sh.order_cap) return DCB_OK;
  pool_free(sh.pool, sh.device, sh.d_order, sh.cap_order);
  sh.d_order = nullptr;
  sh.order_cap = 0;
  uint8_t *p = nullptr;
  CUDA_TRY(pool_alloc(sh.pool, sh.device, std::max<uint64_t>(n, 1024) * 4, &p, &sh.cap_order));
  sh.d_order = reinterpret_cast<uint32_t *>(p);
  sh.order_cap = std::max<uint64_t>(n, 1024);
  return DCB_OK;
}

void tl_mark(dcb_ctx *ctx, const std::string &name, cudaStream_t s, bool begin);

// Pipeline slices: the slice's compressed bytes, on the device's upload stream (slice order = issue order); the
// slice's own stream waits for them.  Issued slice by slice, interleaved with the slices' launches, so that the small
// descriptor copies of slice k are not queued behind the bulk copies of slices k+1.. on the copy engine.
int issue_arena_copy(dcb_ctx *ctx, dcb_batch *b, Shard &sh, int dev_index) {
  if (!sh.arena_pending) return DCB_OK;
  sh.arena_pending = false;
  cudaStream_t st = ctx->streams[dev_index], cs = ctx->copy_in[dev_index];
  CUDA_TRY(cudaSetDevice(sh.device));
  tl_mark(ctx, "h2d s" + std::to_string(dev_index), cs, true);
  CUDA_TRY(cudaMemcpyAsync(sh.d_in + kFrontPad, b->host_arena + sh.direct_lo, sh.direct_hi - sh.direct_lo,
                           cudaMemcpyHostToDevice, cs));
  tl_mark(ctx, "", cs, false);
  CUDA_TRY(cudaEventRecord(ctx->in_ev[dev_index], cs));
  CUDA_TRY(cudaStreamWaitEvent(st, ctx->in_ev[dev_index], 0));
  return DCB_OK;
}

// point order: the explicit faces of an indexed Edgebreaker buffer travel with its maps (the NULL form reads the maps);
// faces in the arena: so do the host-decoded faces of sequential meshes
bool uploads_faces(const Shard &sh, const BufRec &r) {
  if (!r.pt_faces || sh.walks0[r.local].status != DCB_OK) return false;
  return (sh.pts && r.is_eb) || r.face_src == 1;
}

// Mesh connectivity maps (56 bytes per vertex, read by para_deps_kernel only): on the device's upload stream, issued
// BEHIND the first rANS launch of the decode so that the copy hides behind the symbol chains; `st` then waits for it.
// From pageable memory cudaMemcpyAsync stages through the driver and holds the calling thread, not the GPU.
int issue_maps_copy(dcb_ctx *ctx, dcb_batch *b, Shard &sh, int dev_index) {
  if (!sh.maps_pending) return DCB_OK;
  sh.maps_pending = false;
  cudaStream_t st = ctx->streams[dev_index], cs = ctx->copy_in[dev_index];
  CUDA_TRY(cudaSetDevice(sh.device));
  tl_mark(ctx, "h2d maps s" + std::to_string(dev_index), cs, true);
  // Large map sets (configs[3]: 56 MB per million-vertex mesh): the caller's arrays are pageable memory, from which
  // cudaMemcpyAsync runs at a fraction of the link rate and blocks this thread.  A few host threads copy them piece by
  // piece into pinned staging (same layout as the device arena) while the DMA of the finished pieces is already running.
  constexpr uint64_t kMapsStageMin = 32ull << 20, kPiece = 8ull << 20;
  bool staged = false;
  if (sh.maps_bytes >= kMapsStageMin) {
    if (!sh.h_maps && pinned_alloc(sh.pool, sh.maps_bytes, &sh.h_maps, &sh.cap_hmaps) != cudaSuccess) {
      cudaGetLastError();
      sh.h_maps = nullptr;
    }
    if (sh.h_maps) {
      struct Piece { const uint8_t *src; uint64_t off, bytes; };
      std::vector<Piece> pieces;
      try {
        for (int k : sh.bufs)
          for (const MeshMapsHost &m : b->bufs[k].maps)
            if (m.set) {
              const void *src[4] = {m.opposite, m.corner_to_vertex, m.data_to_corner, m.vertex_to_data};
              const uint64_t sz[4] = {m.n_corners * 4, m.n_corners * 4, m.n_entries * 4, m.n_vertices * 4};
              for (int j = 0; j < 4; ++j)
                for (uint64_t o = 0; o < sz[j]; o += kPiece)
                  pieces.push_back({(const uint8_t *)src[j] + o, m.dev_off[j] + o, std::min(kPiece, sz[j] - o)});
            }
        for (int k : sh.bufs)
          if (const BufRec &r = b->bufs[k]; uploads_faces(sh, r))
            for (uint64_t o = 0; o < r.pt_n_faces * 12; o += kPiece)
              pieces.push_back({(const uint8_t *)r.pt_faces + o, r.faces_dev_off + o, std::min(kPiece, r.pt_n_faces * 12 - o)});
        std::unique_ptr<std::atomic<uint8_t>[]> done(new std::atomic<uint8_t>[pieces.size()]);
        for (size_t i = 0; i < pieces.size(); ++i) done[i].store(0, std::memory_order_relaxed);
        std::atomic<size_t> next{0};
        uint8_t *stage = sh.h_maps;
        auto work = [&]() {
          for (size_t i = next.fetch_add(1); i < pieces.size(); i = next.fetch_add(1)) {
            memcpy(stage + pieces[i].off, pieces[i].src, pieces[i].bytes);
            done[i].store(1, std::memory_order_release);
          }
        };
        const unsigned hw = std::max(2u, std::thread::hardware_concurrency());
        const size_t n_threads = std::min<size_t>(std::min<size_t>(8, hw / 2), pieces.size());
        std::vector<std::thread> th;
        th.reserve(n_threads);
        try {
          for (size_t t = 0; t < n_threads; ++t) th.emplace_back(work);
        } catch (...) {  // no more threads to be had: the ones that started (or this one) do the copying
        }
        if (th.empty()) work();
        cudaError_t ce = cudaSuccess;
        for (size_t i = 0; i < pieces.size(); ++i) {
          while (!done[i].load(std::memory_order_acquire)) std::this_thread::yield();
          if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(sh.d_maps + pieces[i].off, stage + pieces[i].off, pieces[i].bytes, cudaMemcpyHostToDevice, cs);
        }
        for (std::thread &t : th) t.join();
        CUDA_TRY(ce);
        staged = true;
      } catch (const std::bad_alloc &) {
        return DCB_ERR_OOM;
      }
    }
  }
  if (!staged)
  for (int k : sh.bufs)
    for (const MeshMapsHost &m : b->bufs[k].maps)
      if (m.set) {
        if (m.n_corners) {
          CUDA_TRY(cudaMemcpyAsync(sh.d_maps + m.dev_off[0], m.opposite, m.n_corners * 4, cudaMemcpyHostToDevice, cs));
          CUDA_TRY(cudaMemcpyAsync(sh.d_maps + m.dev_off[1], m.corner_to_vertex, m.n_corners * 4, cudaMemcpyHostToDevice, cs));
        }
        if (m.n_entries) CUDA_TRY(cudaMemcpyAsync(sh.d_maps + m.dev_off[2], m.data_to_corner, m.n_entries * 4, cudaMemcpyHostToDevice, cs));
        if (m.n_vertices) CUDA_TRY(cudaMemcpyAsync(sh.d_maps + m.dev_off[3], m.vertex_to_data, m.n_vertices * 4, cudaMemcpyHostToDevice, cs));
      }
  if (!staged)
    for (int k : sh.bufs)
      if (const BufRec &r = b->bufs[k]; uploads_faces(sh, r) && r.pt_n_faces)
        CUDA_TRY(cudaMemcpyAsync(sh.d_maps + r.faces_dev_off, r.pt_faces, r.pt_n_faces * 12, cudaMemcpyHostToDevice, cs));
  tl_mark(ctx, "", cs, false);
  CUDA_TRY(cudaEventRecord(ctx->maps_ev[dev_index], cs));
  CUDA_TRY(cudaStreamWaitEvent(st, ctx->maps_ev[dev_index], 0));
  return DCB_OK;
}

// Point order: the job tables of the point stage (dcb_points.cu) -- one map per (Edgebreaker buffer, attributes decoder)
// with attributes, one gather per attribute (identity rows for point clouds and sequential meshes sharing the shard) --
// and the shard's arena for them: entry-order staging | point maps (u32 per point and decoder) | tables.
int plan_points(dcb_batch *b, Shard &sh, cudaStream_t st) {
  std::vector<PointMapJob> mj;
  std::vector<PointGatherJob> gj;
  std::vector<uint64_t> cpre{0}, ppre{0}, upre{0};
  for (size_t bi = 0; bi < sh.walks0.size(); ++bi) {
    const BufWalk &w = sh.walks0[bi];
    const BufRec &r = b->bufs[sh.bufs[bi]];
    if (w.status != DCB_OK) continue;
    std::vector<uint64_t> dec_map(r.is_eb ? r.maps.size() : 0, ~0ull);
    for (int i = 0; i < w.stream_count; ++i) {
      const uint32_t si = (uint32_t)(w.stream_first + i);
      const StreamDesc &s = sh.streams0[si];
      if (sh.fin_bytes[si] == 0) continue;
      uint64_t map_off = ~0ull;
      if (r.is_eb) {
        const MeshMapsHost &m = r.maps[s.decoder_id];
        if (dec_map[s.decoder_id] == ~0ull) {
          PointMapJob j{};
          j.faces_off = r.pt_faces ? r.faces_dev_off : r.maps[0].dev_off[1];
          j.c2v_off = m.dev_off[1];
          j.v2d_off = m.dev_off[3];
          j.map_off = ppre.back();
          j.n_corners = (uint32_t)m.n_corners;
          j.n_points = r.info.n_points;
          j.n_vertices = (uint32_t)m.n_vertices;
          j.n_entries = (uint32_t)m.n_entries;
          j.status_si = (uint32_t)w.stream_first;
          dec_map[s.decoder_id] = j.map_off;
          mj.push_back(j);
          cpre.push_back(cpre.back() + m.n_corners);
          ppre.push_back(ppre.back() + r.info.n_points);
        }
        map_off = dec_map[s.decoder_id];
      }
      PointGatherJob g{};
      g.src_off = s.out_off;
      g.dst_off = sh.fin_off[si];
      g.map_off = map_off;
      g.row_bytes = (uint32_t)row_bytes(s);
      g.rows = (uint32_t)(sh.fin_bytes[si] / g.row_bytes);
      g.st_first = (uint32_t)w.stream_first;
      g.st_count = (uint32_t)w.stream_count;
      while (g.vec_shift < 4 && g.row_bytes % (2u << g.vec_shift) == 0) ++g.vec_shift;
      gj.push_back(g);
      upre.push_back(upre.back() + (uint64_t)g.rows * (g.row_bytes >> g.vec_shift));
    }
  }
  const uint64_t off_pmap = align_up(sh.stage_bytes, 256);
  const uint64_t off_mj = align_up(off_pmap + 4 * ppre.back(), 256);
  const uint64_t off_cpre = align_up(off_mj + mj.size() * sizeof(PointMapJob), 16);
  const uint64_t off_ppre = align_up(off_cpre + cpre.size() * 8, 16);
  const uint64_t off_gj = align_up(off_ppre + ppre.size() * 8, 16);
  const uint64_t off_upre = align_up(off_gj + gj.size() * sizeof(PointGatherJob), 16);
  const uint64_t total = off_upre + upre.size() * 8;
  CUDA_TRY(pool_alloc(sh.pool, sh.device, total, &sh.d_pts, &sh.cap_pts));
  std::vector<uint8_t> &t = sh.pts_tables;  // outlives the asynchronous upload
  t.assign(total - off_mj, 0);
  auto put = [&](uint64_t off, const void *src, uint64_t n) { if (n) memcpy(t.data() + (off - off_mj), src, n); };
  put(off_mj, mj.data(), mj.size() * sizeof(PointMapJob));
  put(off_cpre, cpre.data(), cpre.size() * 8);
  put(off_ppre, ppre.data(), ppre.size() * 8);
  put(off_gj, gj.data(), gj.size() * sizeof(PointGatherJob));
  put(off_upre, upre.data(), upre.size() * 8);
  CUDA_TRY(cudaMemcpyAsync(sh.d_pts + off_mj, t.data(), t.size(), cudaMemcpyHostToDevice, st));
  PointStage &p = sh.pstage;
  p.maps = reinterpret_cast<const PointMapJob *>(sh.d_pts + off_mj);
  p.corner_prefix = reinterpret_cast<const uint64_t *>(sh.d_pts + off_cpre);
  p.point_prefix = reinterpret_cast<const uint64_t *>(sh.d_pts + off_ppre);
  p.n_maps = (uint32_t)mj.size();
  p.gathers = reinterpret_cast<const PointGatherJob *>(sh.d_pts + off_gj);
  p.unit_prefix = reinterpret_cast<const uint64_t *>(sh.d_pts + off_upre);
  p.n_gathers = (uint32_t)gj.size();
  p.pmap = reinterpret_cast<uint32_t *>(sh.d_pts + off_pmap);
  p.pmap_words = ppre.back();
  p.total_corners = cpre.back();
  p.total_units = upre.back();
  p.stage = sh.d_pts;
  return DCB_OK;
}

// DCB_FACES_ARENA: the job tables of the faces stage (dcb_faces.cu) -- one job per mesh buffer with faces: fixed-width
// plain indices from the input arena, u32 faces from the maps arena, varint runs with their checkpoints
int plan_faces(dcb_batch *b, Shard &sh, cudaStream_t st) {
  std::vector<FaceJob> pj, vj, ij;
  std::vector<uint64_t> upre{0}, cpre{0}, ckpt, ipre{0};
  for (uint32_t si = sh.idx_first; si < sh.streams.size(); ++si) {
    BufRec &r = b->bufs[sh.streams[si].buf_index];
    FaceJob f{};
    f.dst_off = r.face_off;
    f.n_idx = 3 * r.n_faces;
    f.stream = si;
    r.idx_job = (int32_t)ij.size();
    ij.push_back(f);
    ipre.push_back(ipre.back() + (f.n_idx + DCB_INDEX_CHUNK - 1) / DCB_INDEX_CHUNK);
  }
  for (int k : sh.bufs) {
    const BufRec &r = b->bufs[k];
    if (!r.face_src || !r.n_faces || r.idx_job >= 0) continue;
    FaceJob f{};
    f.dst_off = r.face_off;
    f.n_idx = 3 * r.n_faces;
    if (r.face_src == 2) {
      f.src_off = r.arena_off + r.seq_loc.off;
      f.width = (uint32_t)r.seq_loc.width;
      f.n_bytes = r.seq_loc.bytes;
    } else {
      f.from_maps = 1;
      f.width = 4;
      f.src_off = r.pt_faces ? r.faces_dev_off : r.maps[0].dev_off[1];
    }
    if (f.width) {
      pj.push_back(f);
      upre.push_back(upre.back() + (f.n_idx + 3) / 4);
    } else {
      f.ckpt_off = ckpt.size();
      ckpt.insert(ckpt.end(), r.seq_loc.ckpt.begin(), r.seq_loc.ckpt.end());
      vj.push_back(f);
      cpre.push_back(cpre.back() + r.seq_loc.ckpt.size());
    }
  }
  FaceStage &p = sh.fstage;
  p = FaceStage{};
  if (pj.empty() && vj.empty() && ij.empty()) return DCB_OK;
  const uint64_t off_pj = 0;
  const uint64_t off_upre = align_up(off_pj + pj.size() * sizeof(FaceJob), 16);
  const uint64_t off_vj = align_up(off_upre + upre.size() * 8, 16);
  const uint64_t off_cpre = align_up(off_vj + vj.size() * sizeof(FaceJob), 16);
  const uint64_t off_ckpt = align_up(off_cpre + cpre.size() * 8, 16);
  const uint64_t off_ij = align_up(off_ckpt + ckpt.size() * 8, 16);
  const uint64_t off_ipre = align_up(off_ij + ij.size() * sizeof(FaceJob), 16);
  const uint64_t n_ich = ipre.back();
  // device-written: chunk sums, minima, maxima (int64 each) and one status per index job
  const uint64_t off_csum = align_up(off_ipre + ipre.size() * 8, 16);
  const uint64_t off_cmin = off_csum + 8 * n_ich, off_cmax = off_cmin + 8 * n_ich, off_stat = off_cmax + 8 * n_ich;
  const uint64_t total = off_stat + 4 * ij.size();
  CUDA_TRY(pool_alloc(sh.pool, sh.device, total, &sh.d_faces, &sh.cap_faces));
  std::vector<uint8_t> &t = sh.faces_tables;  // outlives the asynchronous upload
  t.assign(total, 0);
  auto put = [&](uint64_t off, const void *src, uint64_t n) { if (n) memcpy(t.data() + off, src, n); };
  put(off_pj, pj.data(), pj.size() * sizeof(FaceJob));
  put(off_upre, upre.data(), upre.size() * 8);
  put(off_vj, vj.data(), vj.size() * sizeof(FaceJob));
  put(off_cpre, cpre.data(), cpre.size() * 8);
  put(off_ckpt, ckpt.data(), ckpt.size() * 8);
  put(off_ij, ij.data(), ij.size() * sizeof(FaceJob));
  put(off_ipre, ipre.data(), ipre.size() * 8);
  CUDA_TRY(cudaMemcpyAsync(sh.d_faces, t.data(), off_csum, cudaMemcpyHostToDevice, st));
  if (!ij.empty() && (!sh.h_fstatus || sh.cap_hfstatus < 4 * ij.size())) {
    if (sh.h_fstatus) pinned_free(sh.pool, sh.h_fstatus, sh.cap_hfstatus);
    uint8_t *hp = nullptr;
    CUDA_TRY(pinned_alloc(sh.pool, 4 * ij.size(), &hp, &sh.cap_hfstatus));
    sh.h_fstatus = reinterpret_cast<int32_t *>(hp);
  }
  p.plain = reinterpret_cast<const FaceJob *>(sh.d_faces + off_pj);
  p.unit_prefix = reinterpret_cast<const uint64_t *>(sh.d_faces + off_upre);
  p.n_plain = (uint32_t)pj.size();
  p.varint = reinterpret_cast<const FaceJob *>(sh.d_faces + off_vj);
  p.chunk_prefix = reinterpret_cast<const uint64_t *>(sh.d_faces + off_cpre);
  p.n_varint = (uint32_t)vj.size();
  p.ckpt = reinterpret_cast<const uint64_t *>(sh.d_faces + off_ckpt);
  p.total_units = upre.back();
  p.total_chunks = cpre.back();
  p.index = reinterpret_cast<const FaceJob *>(sh.d_faces + off_ij);
  p.index_prefix = reinterpret_cast<const uint64_t *>(sh.d_faces + off_ipre);
  p.n_index = (uint32_t)ij.size();
  p.total_index_chunks = n_ich;
  p.chunk_sum = reinterpret_cast<int64_t *>(sh.d_faces + off_csum);
  p.chunk_min = reinterpret_cast<int64_t *>(sh.d_faces + off_cmin);
  p.chunk_max = reinterpret_cast<int64_t *>(sh.d_faces + off_cmax);
  p.status = reinterpret_cast<int32_t *>(sh.d_faces + off_stat);
  return DCB_OK;
}

// DCB_FACES_ARENA: fills the faces regions of a shard, on its stream behind its decode (the maps copy first)
int faces_shard(dcb_ctx *ctx, dcb_batch *b, Shard &sh, int dev_index, uint8_t *d_out) {
  if (!sh.fstage.total_units && !sh.fstage.total_chunks && !sh.fstage.n_index) return DCB_OK;
  int rc = issue_maps_copy(ctx, b, sh, dev_index);
  if (rc) return rc;
  cudaStream_t st = ctx->streams[dev_index];
  CUDA_TRY(cudaSetDevice(sh.device));
  tl_mark(ctx, "faces s" + std::to_string(dev_index), st, true);
  // behind the joins of decode_shard: the Raw index streams have left their symbols in the scratch
  DevArenas A{sh.d_in, d_out, nullptr, sh.d_aux, nullptr, sh.d_maps};
  CUDA_TRY(dcb_launch_faces(sh.fstage, sh.d_streams, A, (uint32_t)ctx->num_sms[dev_index], st));
  tl_mark(ctx, "", st, false);
  if (sh.fstage.n_index)  // per-buffer verdicts of the index scan, folded in by collect_status after the caller's sync
    CUDA_TRY(cudaMemcpyAsync(sh.h_fstatus, sh.fstage.status, 4ull * sh.fstage.n_index, cudaMemcpyDeviceToHost, st));
  dcb_launch_stats &stats = dev_index == 0 ? ctx->stats : ctx->dev_stats[dev_index];
  stats.n_launches += (sh.fstage.total_units ? 1 : 0) + (sh.fstage.total_chunks ? 1 : 0) + (sh.fstage.n_index ? 3 : 0);
  return DCB_OK;
}

int upload_shard(dcb_ctx *ctx, dcb_batch *b, Shard &sh, int dev_index) {
  if (sh.uploaded) return DCB_OK;
  cudaStream_t st = ctx->streams[dev_index];
  CUDA_TRY(cudaSetDevice(sh.device));
  sh.pool = ctx->pool;
  CUDA_TRY(pool_alloc(sh.pool, sh.device, sh.in_bytes, &sh.d_in, &sh.cap_in));
  CUDA_TRY(cudaMemsetAsync(sh.d_in, 0, kFrontPad, st));
  CUDA_TRY(cudaMemsetAsync(sh.d_in + sh.in_bytes - kBackPad, 0, kBackPad, st));
  if (sh.direct && sh.share > 1) {
    sh.arena_pending = true;  // pipeline slices: issue_arena_copy, right before the slice's kernels are launched
  } else if (sh.direct) {
    CUDA_TRY(cudaMemcpyAsync(sh.d_in + kFrontPad, b->host_arena + sh.direct_lo, sh.direct_hi - sh.direct_lo,
                             cudaMemcpyHostToDevice, st));
  } else if (!sh.bufs.empty()) {
    CUDA_TRY(pinned_alloc(sh.pool, sh.in_bytes, &sh.h_stage, &sh.cap_stage));
    for (int k : sh.bufs) memcpy(sh.h_stage + b->bufs[k].arena_off, b->bufs[k].src, b->bufs[k].len);
    CUDA_TRY(cudaMemcpyAsync(sh.d_in + kFrontPad, sh.h_stage + kFrontPad, sh.in_bytes - kFrontPad - kBackPad,
                             cudaMemcpyHostToDevice, st));
  }
  // mesh maps: laid out and allocated here, copied by issue_maps_copy (behind the first rANS launch of the decode)
  uint64_t mbytes = 0;
  for (int k : sh.bufs)
    for (MeshMapsHost &m : b->bufs[k].maps)
      if (m.set) {
        const uint64_t sz[4] = {m.n_corners, m.n_corners, m.n_entries, m.n_vertices};
        for (int j = 0; j < 4; ++j) {
          m.dev_off[j] = mbytes;
          mbytes = align_up(mbytes + sz[j] * 4, 16);
        }
      }
  for (int k : sh.bufs)  // point order: explicit faces travel with the maps
    if (BufRec &r = b->bufs[k]; uploads_faces(sh, r)) {
      r.faces_dev_off = mbytes;
      mbytes = align_up(mbytes + r.pt_n_faces * 12, 16);
    }
  sh.maps_bytes = mbytes;
  if (mbytes) {
    CUDA_TRY(pool_alloc(sh.pool, sh.device, mbytes, &sh.d_maps, &sh.cap_maps));
    sh.maps_pending = true;
    for (int k : sh.bufs) {
      const BufRec &r = b->bufs[k];
      const BufWalk &w = sh.walks0[r.local];
      for (int i = 0; i < w.stream_count; ++i) {
        for (std::vector<StreamDesc> *vs : {&sh.streams0, &sh.streams}) {
          StreamDesc &s = (*vs)[w.stream_first + i];
          if (s.has_maps && s.decoder_id < r.maps.size())
            for (int j = 0; j < 4; ++j) s.map_off[j] = r.maps[s.decoder_id].dev_off[j];
        }
      }
    }
  }
  // every allocation of a decode happens here, before any kernel is launched: a cudaMalloc issued between two
  // launches keeps them from running concurrently (pipeline slices, side streams)
  {
    int rc = ensure_order(sh, 4 * (uint64_t)sh.streams.size() + sh.bufs.size() + 1024);
    if (rc) return rc;
  }
  if (!sh.streams.empty()) {
    uint8_t *p = nullptr;
    CUDA_TRY(pool_alloc(sh.pool, sh.device, sh.streams.size() * sizeof(StreamDesc), &p, &sh.cap_streams));
    sh.d_streams = reinterpret_cast<StreamDesc *>(p);
  }
  if (!sh.walks.empty()) {
    uint8_t *p = nullptr;
    CUDA_TRY(pool_alloc(sh.pool, sh.device, sh.walks.size() * sizeof(BufWalk), &p, &sh.cap_walks));
    sh.d_walks = reinterpret_cast<BufWalk *>(p);
  }
  if (!sh.h_desc && !sh.streams.empty())
    CUDA_TRY(pinned_alloc(sh.pool, sh.streams.size() * sizeof(StreamDesc) + sh.walks.size() * sizeof(BufWalk) + 16, &sh.h_desc,
                          &sh.cap_hdesc));
  if (sh.aux_bytes) {
    CUDA_TRY(pool_alloc(sh.pool, sh.device, sh.aux_bytes, &sh.d_aux, &sh.cap_aux));
    CUDA_TRY(cudaMemsetAsync(sh.d_aux, 0, sh.aux_bytes, st));  // look-back words start with epoch 0 (never a live epoch)
  }
  if (sh.pts) {
    int rc = plan_points(b, sh, st);
    if (rc) return rc;
  }
  if (b->faces == DCB_FACES_ARENA) {
    int rc = plan_faces(b, sh, st);
    if (rc) return rc;
  }
  sh.uploaded = true;
  sh.dirty = true;
  return DCB_OK;
}

// look-back epochs cycle through 1 .. 2^30 - 1: the words carry 30 bits of it and zeroed scratch must never look live
inline uint32_t next_epoch(Shard &sh) {
  sh.epoch = sh.epoch >= 0x3FFFFFFEu ? 1u : sh.epoch + 1u;
  return sh.epoch;
}

// Stream descriptors and walks as the device left them (statuses, bits_total, the PRED_DATA / XFORM_PARAMS the resumed
// walks parsed) travel back through pinned memory on the shard's stream; absorb_descs folds them into the host copies
// once the caller has synchronised.  Nothing here blocks the host thread.
int queue_desc_copyback(dcb_ctx *ctx, Shard &sh, cudaStream_t st) {
  const uint64_t nb_s = sh.streams.size() * sizeof(StreamDesc), nb_w = sh.walks.size() * sizeof(BufWalk);
  if (!sh.h_desc) CUDA_TRY(pinned_alloc(sh.pool, nb_s + nb_w + 16, &sh.h_desc, &sh.cap_hdesc));
  CUDA_TRY(cudaMemcpyAsync(sh.h_desc, sh.d_streams, nb_s, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(sh.h_desc + nb_s, sh.d_walks, nb_w, cudaMemcpyDeviceToHost, st));
  sh.desc_pending = true;
  sh.dirty = true;
  (void)ctx;
  return DCB_OK;
}
void absorb_descs(dcb_batch *b) {
  for (Shard &sh : b->shards) {
    if (!sh.desc_pending) continue;
    const uint64_t nb_s = sh.streams.size() * sizeof(StreamDesc), nb_w = sh.walks.size() * sizeof(BufWalk);
    memcpy(sh.streams.data(), sh.h_desc, nb_s);
    memcpy(sh.walks.data(), sh.h_desc + nb_s, nb_w);
    sh.desc_pending = false;
  }
}

// fresh descriptors: the decode must not depend on what an earlier decode left behind
int reset_descriptors(Shard &sh, cudaStream_t st) {
  if (sh.dirty) {
    sh.streams = sh.streams0;
    sh.walks = sh.walks0;
    CUDA_TRY(cudaMemcpyAsync(sh.d_streams, sh.streams.data(), sh.streams.size() * sizeof(StreamDesc), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(sh.d_walks, sh.walks.data(), sh.walks.size() * sizeof(BufWalk), cudaMemcpyHostToDevice, st));
    sh.dirty = false;
  }
  sh.tags_launched.assign(sh.streams.size(), 0);
  return DCB_OK;
}

// what the launches of one decode of a shard share
struct ShardRun {
  dcb_ctx *ctx;
  dcb_batch *b;
  Shard &sh;
  int dev_index;
  cudaStream_t st;  // the shard's stream
  uint32_t num_sms;
  dcb_launch_stats &stats;
  DevArenas A;
  uint32_t dump;
  bool events;      // a timed decode on context device 0: records ctx->ev[] and the algorithm bytes
  bool dbg_tl;      // DCB_DEBUG_TIMING spans of this decode
  bool side_used[3] = {false, false, false};
  // a DCB_DEBUG_TIMING span on stream s: begun with a name, ended without one
  void tl(cudaStream_t s, const char *begin = nullptr) const {
    if (dbg_tl) tl_mark(ctx, begin ? std::string(begin) + " s" + std::to_string(dev_index) : std::string(), s, begin != nullptr);
  }
};

// DCB_DEBUG_PLAN: the planner's choices for one rANS group
void print_plan(const Group &g) {
  if (!env_flags().debug_plan) return;
  fprintf(stderr, "[dcb plan] %s group ncp=%d wide=%d compact=%u prec=%u entries=%u mode=%u zig=%u: %u streams, %llu symbols, "
                  "k=%u lut=%uB lutb=%uB ent=%uB lanes=%u pairs=%u split=%u direct=%u global=%d rec_ka=%u rec=%uB (need x8: %u %u %u %u, exc %u)\n",
          g.tag ? "tag" : "raw", g.ncp, (int)g.wide, g.compact, g.prec_bits, g.entries, g.mode, g.zig, (uint32_t)g.order.size(),
          (unsigned long long)g.total_symbols, g.lut_shift, g.lut_bytes, g.lutb_bytes, g.ent_bytes, g.lanes, g.pairs, g.split,
          g.direct, (int)g.table_global, g.rec_ka, g.rec_bytes, g.rec_max[0], g.rec_max[1], g.rec_max[2], g.rec_max[3], g.exc_all);
}

// the launch of a planned group over n of its streams, listed at d_order
RansLaunch rans_launch(const Group &g, StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t dump) {
  return RansLaunch{d_streams, d_order, n, g.lanes, g.lut_bytes, g.lutb_bytes, g.ent_bytes, g.entries, g.rec_ka ? g.exc_all : g.exc,
                    g.lut_shift, g.prec_bits, dump, g.compact, g.zig, g.mode, g.pairs, g.direct, g.rec_ka, g.rec_bytes, g.split};
}

// Walks blocked on their last stream, a Tagged one, finished on the host: their streams' kernels follow from header
// fields the host already has.
void finish_tagged_walks(Shard &sh, const std::vector<uint32_t> &blocked) {
  for (uint32_t bi : blocked) {
    BufWalk &w = sh.walks[bi];
    for (int i = 0; i < w.stream_count; ++i) {
      StreamDesc &s = sh.streams[w.stream_first + i];
      if (s.state == ST_READY) continue;
      if (s.state == ST_TAGS_PENDING) {
        bool has_scheme, mesh_scheme;
        int e;
        walk_scheme_kind(w, s, has_scheme, mesh_scheme, e);
        s.recon = !has_scheme ? (uint8_t)RECON_NONE
                  : s.transform == XF_WRAP ? (uint8_t)(mesh_scheme ? RECON_PARA_WRAP : RECON_DELTA_WRAP)
                  : s.transform == XF_OCT_CANON ? (uint8_t)(mesh_scheme ? RECON_GEO_OCT_CANON : RECON_DELTA_OCT_CANON)
                                                : (uint8_t)(mesh_scheme ? RECON_GEO_OCT : RECON_DELTA_OCT);
      }
      if (s.seq_type == SEQ_QUANTIZATION) s.store = STORE_DEQUANT;
      else if (s.seq_type == SEQ_NORMALS) s.store = STORE_OCT_UNIT;
      else if (s.seq_type == SEQ_INTEGER) s.store = STORE_NARROW;
      s.state = ST_READY;
    }
    w.blocked = -1;
    w.phase = 2;
  }
}

// Tagged streams: decode tags, resume the walks behind their bit areas, round by round.  `deferred`: the last round's
// walks were finished on the host (finish_tagged_walks); the device descriptors hold what their resumed walks found.
int run_tag_rounds(ShardRun &r, bool &deferred) {
  dcb_ctx *ctx = r.ctx;
  Shard &sh = r.sh;
  const cudaStream_t st = r.st;
  for (;;) {
    Group g{};
    g.tag = true; g.ncp = 1; g.compact = 1; g.prec_bits = 12;
    std::vector<uint32_t> blocked;
    for (size_t bi = 0; bi < sh.walks.size(); ++bi) {
      const BufWalk &w = sh.walks[bi];
      if (w.status != DCB_OK || w.blocked < 0) continue;
      const uint32_t si = (uint32_t)(w.stream_first + w.blocked);
      if (sh.tags_launched[si]) continue;
      sh.tags_launched[si] = 1;
      g.order.push_back(si);
      g.entries = std::max(g.entries, sh.streams[si].n_active);
      g.exc = std::max(g.exc, sh.streams[si].n_active - std::min(sh.streams[si].n_active, sh.streams[si].dense_prefix));
      g.total_symbols += sh.streams[si].n_entries;
      g.note_table(sh.streams[si]);
      blocked.push_back((uint32_t)bi);
    }
    if (g.order.empty()) return DCB_OK;
    sh.dirty = true;
    std::stable_sort(g.order.begin(), g.order.end(),
                     [&](uint32_t x, uint32_t y) { return sh.streams[x].n_entries > sh.streams[y].n_entries; });
    std::vector<Group *> gs{&g};
    plan_rans_groups(gs, r.num_sms, (uint32_t)sh.share);
    if (g.table_global) return DCB_ERR_STATE;  // cannot happen: tag alphabets are tiny (<= 2^24 guarded by table size)
    print_plan(g);
    int rc = ensure_order(sh, g.order.size() + blocked.size());
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(sh.d_order, g.order.data(), g.order.size() * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(sh.d_order + g.order.size(), blocked.data(), blocked.size() * 4, cudaMemcpyHostToDevice, st));
    const RansLaunch L = rans_launch(g, sh.d_streams, sh.d_order, (uint32_t)g.order.size(), r.dump);
    const bool time_tag = r.events && !ctx->ev_tag;
    if (time_tag) {
      CUDA_TRY(cudaEventRecord(ctx->ev[4], st));
      for (uint32_t si : g.order) ctx->algo_tag += sh.streams[si].payload_len + sh.streams[si].n_entries;
    }
    CUDA_TRY(g.rec_ka ? dcb_launch_rans_tag_rec(L, r.A, st) : g.pairs ? dcb_launch_rans_tag_pc(L, r.A, st) : dcb_launch_rans_tag(L, r.A, st));
    if (time_tag) {
      CUDA_TRY(cudaEventRecord(ctx->ev[5], st));
      ctx->ev_tag = true;
    }
    rc = issue_maps_copy(ctx, r.b, sh, r.dev_index);  // the maps travel while the tag chains run
    if (rc) return rc;
    CUDA_TRY(dcb_launch_resolve(r.A, sh.d_walks, sh.d_order + g.order.size(), (uint32_t)blocked.size(), sh.d_streams, st));
    r.stats.n_launches += 2;
    r.stats.n_streams += (int32_t)g.order.size();
    // Nothing follows a Tagged attribute that closes its buffer, so the host does not need what the resumed walk finds
    // (wrap bounds, quantisation parameters: they stay in the device descriptors, where the kernels read them) -- only
    // WHICH kernels to launch, and that follows from the header fields it already has.  No round trip then.
    bool all_last = !env_flags().no_fast_tagged;
    for (uint32_t bi : blocked) all_last = all_last && sh.walks[bi].blocked == sh.walks[bi].stream_count - 1;
    if (all_last) {
      finish_tagged_walks(sh, blocked);
      deferred = true;
      return DCB_OK;
    }
    CUDA_TRY(cudaMemcpyAsync(sh.streams.data(), sh.d_streams, sh.streams.size() * sizeof(StreamDesc), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(sh.walks.data(), sh.d_walks, sh.walks.size() * sizeof(BufWalk), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
}

constexpr int kWideAttrMode = 5;  // RawKey::mode of wide attributes: a group of their own, launched in mode 0

// Sort the ready streams of a shard into its launches and plan them.  Host work only: it makes no CUDA call.  Wide
// attributes it cannot decode get DCB_ERR_UNSUPPORTED in sh.streams.
int plan_shard(const dcb_batch *b, Shard &sh, uint32_t num_sms, ShardPlan &p) {
  p = ShardPlan{};
  // group key of a Raw stream; force_compact: -1 the natural table representation (compact when fewer than half of the
  // alphabet is in use), 0 / 1 dense / compact
  auto raw_key_of = [&](const StreamDesc &s, bool raw_normals, int force_compact) -> RawKey {
    RawKey key;
    key.ncp = s.ncp;
    key.compact = force_compact >= 0 ? force_compact : ((2ull * s.n_active + 1 < s.num_symbols) ? 1 : 0);
    key.prec = s.prec_bits;
    const uint32_t entries = key.compact ? s.n_active : s.num_symbols;
    key.wide = (s.prec_bits > 15 || s.num_symbols > 65535u || (uint64_t)entries * (key.compact ? 4 : 2) + 4 > 60000u) ? 1 : 0;
    key.size_class = (int)ceil_log2(std::max(16u, entries));
    key.zig = s.zigzag ? 1 : 0;
    key.mode = 0;
    if (s.recon == RECON_DELTA_WRAP && s.store == STORE_DEQUANT) key.mode = 1;
    else if (s.recon == RECON_DELTA_WRAP && s.store == STORE_NARROW && dcb_dtype_len(s.data_type) == 1) key.mode = 2;
    else if (raw_normals) key.mode = 3;
    else if (s.recon == RECON_PARA_WRAP && s.zigzag) key.mode = 4;
    return key;
  };
  auto is_raw_normals = [](const StreamDesc &s) {
    // (geometric normals too: the rANS kernel leaves corrections either way; oct_chain / oct_unit skip those streams)
    return s.scheme == SCHEME_RAW && s.ncp == 2 && s.store == STORE_OCT_UNIT &&
           (s.recon == RECON_DELTA_OCT || s.recon == RECON_DELTA_OCT_CANON || s.recon == RECON_GEO_OCT || s.recon == RECON_GEO_OCT_CANON);
  };
  std::map<RawKey, size_t> raw_count;  // streams per natural key
  for (size_t bi = 0; bi < sh.walks.size(); ++bi) {
    const BufWalk &w = sh.walks[bi];
    if (w.status != DCB_OK) continue;
    for (int i = 0; i < w.stream_count; ++i) {
      const StreamDesc &s = sh.streams[(size_t)w.stream_first + i];
      if (s.state == ST_READY && s.scheme == SCHEME_RAW && s.n_entries > 0) raw_count[raw_key_of(s, is_raw_normals(s), -1)]++;
    }
  }
  std::map<RawKey, Group> raw;
  // a Raw stream joins the group of its key; the symbols of a stream are n_entries * ncp one-component ones
  auto add_raw = [&](const RawKey &key, uint32_t si) {
    const StreamDesc &s = sh.streams[si];
    Group &g = raw[key];
    if (g.order.empty()) {
      g.ncp = key.ncp; g.wide = key.wide != 0; g.compact = (uint32_t)key.compact; g.prec_bits = (uint32_t)key.prec;
      g.zig = (uint32_t)key.zig;
      g.force_single_warp = key.mode == kWideAttrMode;
      g.mode = g.force_single_warp ? 0u : (uint32_t)key.mode;
    }
    g.entries = std::max(g.entries, key.compact ? s.n_active : s.num_symbols);
    if (key.compact) g.exc = std::max(g.exc, s.n_active - std::min(s.n_active, s.dense_prefix));
    g.total_symbols += (uint64_t)s.n_entries * s.ncp;
    g.max_entries = std::max(g.max_entries, s.n_entries);
    g.note_table(s);
    g.order.push_back(si);
  };
  for (size_t bi = 0; bi < sh.walks.size(); ++bi) {
    const BufWalk &w = sh.walks[bi];
    if (w.status != DCB_OK) continue;
    for (int i = 0; i < w.stream_count; ++i) {
      const uint32_t si = (uint32_t)(w.stream_first + i);
      const StreamDesc &s = sh.streams[si];
      if (s.state != ST_READY) continue;
      if (s.scheme == SCHEME_GENERIC) {
        p.copy.order.push_back(si);
        p.copy.max_bytes = std::max(p.copy.max_bytes, s.out_bytes);
        continue;
      }
      if (s.n_entries == 0) continue;
      if (s.ncp > 4) {
        // wide integer attribute: a Raw source decodes as n * nc one-component symbols into the scratch (the fused
        // kernel's generic instantiation), then -- as for Tagged and uncompressed sources -- wide_post_kernel
        // reconstructs and stores entry by entry with a run-time component count
        if ((uint64_t)s.n_entries * s.ncp > 0xFFFFFFF0ull || (s.recon != RECON_NONE && s.recon != RECON_DELTA_WRAP)) {
          sh.streams[si].status = DCB_ERR_UNSUPPORTED;
          continue;
        }
        if (s.scheme == SCHEME_RAW) {
          RawKey key = raw_key_of(s, false, -1);
          key.ncp = 1;
          key.mode = kWideAttrMode;
          add_raw(key, si);
        }
        p.wide.order.push_back(si);
        continue;
      }
      // normals behind a Raw stream: the rANS kernel leaves corrections, oct_chain + oct_unit follow on its stream
      const bool raw_normals = is_raw_normals(s);
      const bool geo_normals = s.recon == RECON_GEO_OCT || s.recon == RECON_GEO_OCT_CANON;
      if (geo_normals) {  // geo_normal_kernel finishes the attribute behind the parallelogram kernels of its parent
        p.geo.order.push_back(si);
        p.geo.max_entries = std::max(p.geo.max_entries, s.n_entries);
        p.has_para = true;
      } else if (s.store == STORE_OCT_UNIT && !raw_normals) {
        p.octs.order.push_back(si);
        p.octs.max_entries = std::max(p.octs.max_entries, s.n_entries);
      }
      if (s.scheme == SCHEME_RAW) {
        RawKey key = raw_key_of(s, raw_normals, -1);
        if (!key.compact) {
          // a few streams whose tables came out dense next to a machine-filling group of compact tables of the same
          // shape: they join it (a compact table is always a valid representation) instead of forming a launch of
          // their own that outlasts the big one (uniform LUT with a search loop: 220 instead of 177 cycles per symbol)
          const RawKey twin = raw_key_of(s, raw_normals, 1);
          const auto it_t = raw_count.find(twin), it_n = raw_count.find(key);
          if (it_t != raw_count.end() && it_t->second >= (size_t)num_sms * 8 && it_n->second < (size_t)num_sms) key = twin;
        }
        add_raw(key, si);
      } else if (s.recon == RECON_NONE || s.recon == RECON_DELTA_WRAP || s.recon == RECON_PARA_WRAP || (geo_normals && s.ncp == 2) ||
                 ((s.recon == RECON_DELTA_OCT || s.recon == RECON_DELTA_OCT_CANON) && s.ncp == 2 && s.store == STORE_OCT_UNIT)) {
        // Tagged / uncompressed source: point-parallel extraction; scan-able reconstructions finish there, octahedral
        // corrections go to the scratch and oct_chain_kernel runs the recurrence (as behind a Raw source)
        p.par[s.ncp].max_entries = std::max(p.par[s.ncp].max_entries, s.n_entries);
        p.par[s.ncp].order.push_back(si);
        if (s.recon == RECON_DELTA_WRAP) p.pp[s.ncp].delta = true;
        if (s.recon == RECON_DELTA_OCT || s.recon == RECON_DELTA_OCT_CANON) p.octc.order.push_back(si);
      } else {
        p.post[s.ncp].order.push_back(si);
      }
      if (s.recon == RECON_PARA_WRAP && s.pred_method == PRED_TEX_COORDS_PORTABLE) {
        p.tex.order.push_back(si);
        p.tex.max_entries = std::max(p.tex.max_entries, s.n_entries);
        p.has_para = true;
      } else if (s.recon == RECON_PARA_WRAP && s.pred_method == PRED_CONSTRAINED_MULTI) {
        p.cmp[s.ncp].order.push_back(si);
        p.cmp[s.ncp].max_entries = std::max(p.cmp[s.ncp].max_entries, s.n_entries);
        p.has_para = true;
      } else if (s.recon == RECON_PARA_WRAP) {
        p.para[s.ncp].order.push_back(si);
        p.para[s.ncp].max_entries = std::max(p.para[s.ncp].max_entries, s.n_entries);
        p.has_para = true;
      }
    }
  }
  // Raw index differences of sequential meshes (DCB_FACES_ARENA): one-component streams without zig-zag; they depend on
  // nothing else in their buffer, so their group runs beside the attribute groups (side streams when there are several)
  for (uint32_t si = sh.idx_first; si < sh.streams.size(); ++si) {
    const StreamDesc &s = sh.streams[si];
    if (s.status || sh.walks[b->bufs[s.buf_index].local].status != DCB_OK) continue;
    add_raw(raw_key_of(s, false, -1), si);
  }
  for (auto &kv : raw) p.raw.push_back(std::move(kv.second));
  // the groups run one after another on the shard's stream: each one may use the whole SM
  for (const Group &g : p.raw) p.side_followers = p.side_followers || (g.mode == 3 && p.raw.size() > 1);
  for (Group &g : p.raw) {
    // A handful of outlier streams next to a machine-filling group (one cloud of a batch whose table came out dense)
    // must stay small: the direct slot LUT wants ~50 KB per stream, finds no room beside the big group's CTAs and would
    // run BEHIND it (measured: +17 ms on a 27 ms step); with the two-level tables it runs beside it, on a side stream.
    g.no_direct = g.force_single_warp;
    for (const Group &o : p.raw)
      if (&o != &g && o.order.size() >= (size_t)num_sms * 8) g.no_direct = true;
    std::vector<Group *> one{&g};
    plan_rans_groups(one, num_sms, (uint32_t)sh.share, p.side_followers ? 6u * 1024u : 0u);
  }
  auto longest_first = [&](std::vector<uint32_t> &order) {
    std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return sh.streams[x].n_entries > sh.streams[y].n_entries; });
  };
  for (size_t i = 0; i < p.raw.size(); ++i) {
    longest_first(p.raw[i].order);
    if (p.dom < 0 || p.raw[i].total_symbols > p.raw[p.dom].total_symbols) p.dom = (int)i;
  }
  // par_post2_kernel: per group the run prefix of its streams (runs of run_len chunks) and one ticket word
  for (int n = 1; n <= 4; ++n) {
    Stage &par = p.par[n];
    ShardPlan::ParPost &pp = p.pp[n];
    if (par.order.empty()) continue;
    // longest streams first: whole-stream runs are handed out by ticket, longest-processing-time first
    longest_first(par.order);
    uint64_t total_chunks = 0, max_chunks = 0;
    for (uint32_t si : par.order) {
      const uint64_t nch = ((uint64_t)sh.streams[si].n_entries + DCB_TAG_CHUNK - 1) / DCB_TAG_CHUNK;
      total_chunks += nch;
      max_chunks = std::max(max_chunks, nch);
    }
    dcb_par_post_plan((uint32_t)par.order.size(), total_chunks, (uint32_t)std::min<uint64_t>(max_chunks, 0xFFFFFFFFull),
                      pp.delta, num_sms, n, (uint32_t)sh.share, &pp.run_len, &pp.claim);
    // Chunk-sized runs that look back (delta streams) are ticketed ROUND by round -- chunk r of every stream that has
    // one, then chunk r + 1 -- so that the chunks a warp claims together, and the chunks of neighbouring claims, belong
    // to different streams: in stream-major order a claim's look-back waits for the previous claim's LAST chunk, which
    // waits for that claim's first look-back, and a stream decodes chunk after chunk (measured: 195 ms instead of ~8
    // for 2,000 streams of 100,000 points).  The prefix then runs over rounds: the streams are sorted by length, so
    // round r holds the first count(r) of them.
    if (pp.run_len == 1 && pp.delta && max_chunks <= (1ull << 24)) {
      pp.rounds = (uint32_t)max_chunks;
      pp.runs.assign((size_t)max_chunks + 2, 0u);
      // count(r) = streams with more than r chunks; runs[r + 1] - runs[r] = count(r)
      for (uint32_t si : par.order) {
        const uint64_t nch = ((uint64_t)sh.streams[si].n_entries + DCB_TAG_CHUNK - 1) / DCB_TAG_CHUNK;
        if (nch > 0) pp.runs[(size_t)nch] += 1;  // streams that END after round nch - 1
      }
      if (total_chunks > 0xFFFFFFF0ull) return DCB_ERR_UNSUPPORTED;
      uint64_t alive = par.order.size(), acc = 0;
      for (uint64_t r = 0; r <= max_chunks; ++r) {
        const uint32_t ending = pp.runs[(size_t)r];  // streams with exactly r chunks: gone from round r on
        alive -= ending;
        pp.runs[(size_t)r] = (uint32_t)acc;
        acc += alive;
      }
      pp.runs[(size_t)max_chunks + 1] = 0u;  // the ticket
    } else {
      pp.runs.reserve(par.order.size() + 2);
      uint64_t acc = 0;
      for (uint32_t si : par.order) {
        pp.runs.push_back((uint32_t)acc);
        const uint64_t nch = ((uint64_t)sh.streams[si].n_entries + DCB_TAG_CHUNK - 1) / DCB_TAG_CHUNK;
        acc += (nch + pp.run_len - 1) / pp.run_len;
      }
      if (acc > 0xFFFFFFF0ull) return DCB_ERR_UNSUPPORTED;
      pp.runs.push_back((uint32_t)acc);
      pp.runs.push_back(0u);  // the ticket
    }
  }
  // the device order array: each list's offset is where it lands
  auto append = [&](const std::vector<uint32_t> &v, uint64_t &off) {
    off = p.order.size();
    p.order.insert(p.order.end(), v.begin(), v.end());
  };
  for (Group &g : p.raw) append(g.order, g.order_off);
  for (int n = 1; n <= 4; ++n)
    for (Stage *l : {&p.post[n], &p.para[n], &p.cmp[n], &p.par[n]}) append(l->order, l->order_off);
  for (Stage *l : {&p.copy, &p.octs, &p.octc, &p.tex, &p.geo, &p.wide}) append(l->order, l->order_off);
  for (int n = 1; n <= 4; ++n) append(p.pp[n].runs, p.pp[n].runs_off);
  return DCB_OK;
}

// statistics and kernel name of the decode: those of its dominant Raw group
void note_dominant(ShardRun &r, const Group &g) {
  dcb_ctx *ctx = r.ctx;
  dcb_launch_stats &stats = r.stats;
  const uint32_t n = (uint32_t)g.order.size();
  for (uint32_t si : g.order) {
    const StreamDesc &sd = r.sh.streams[si];
    ctx->algo_raw += (sd.payload_off + sd.payload_len - sd.table_off) + sd.out_bytes;
  }
  stats.lanes_per_warp = (int32_t)g.lanes;
  stats.smem_per_stream = (uint64_t)g.lut_bytes + g.lutb_bytes + g.ent_bytes + DCB_RING_BYTES;
  const RansLaunch Ls = rans_launch(g, nullptr, nullptr, n, 0);
  const uint32_t cta_smem = (g.rec_ka ? dcb_rans_rec_smem_bytes(Ls, 4u * (uint32_t)g.ncp)
                             : g.pairs ? dcb_rans_pc_smem_bytes(Ls, 4u * (uint32_t)g.ncp) : dcb_rans_smem_bytes(Ls, g.table_global)) + kSmemPerCtaReserve;
  const uint64_t per_wave = (uint64_t)r.num_sms * std::max<uint32_t>(1u, std::min<uint32_t>(32u, (kSmemPerSM + 1024u) / cta_smem)) * g.lanes * std::max(1u, g.pairs);
  stats.n_waves = g.table_global ? 1 : (int32_t)((n + per_wave - 1) / per_wave);
  if (g.rec_ka)
    snprintf(ctx->raw_name, sizeof ctx->raw_name, "rans_raw_rec<ncp=%d,u16,smem,mode=%u,bucket records 2^%u|16|1,%ux%u lanes,%uB>", g.ncp,
             g.mode, g.rec_ka, g.pairs, g.lanes, g.rec_bytes);
  else if (g.pairs)
    snprintf(ctx->raw_name, sizeof ctx->raw_name, "rans_raw_pc<ncp=%d,u16,smem,mode=%u,%s,%s,%ux%u lanes>", g.ncp, g.mode,
             g.direct ? "direct slot LUT" : "two-level LUT", g.compact ? "compact" : "dense", g.pairs, g.lanes);
  else
    snprintf(ctx->raw_name, sizeof ctx->raw_name, "rans_raw_fused<ncp=%d,%s,%s,mode=%u,k=%u,%s>", g.ncp,
             g.wide ? "u32" : "u16", g.table_global ? "global" : "smem", g.mode, g.lut_shift,
             g.compact ? "compact" : "dense");
}

// The Raw rANS groups.  `flags_early`: the flag kernels follow on side streams, so those fork too.
int launch_rans_groups(ShardRun &r, const ShardPlan &p, bool flags_early) {
  dcb_ctx *ctx = r.ctx;
  Shard &sh = r.sh;
  const int d = r.dev_index;
  // independent smem-table groups go to side streams so that their chains overlap (c3: positions, normals, colours)
  const bool fan_out = p.raw.size() > 1;
  if (fan_out || flags_early) {
    CUDA_TRY(cudaEventRecord(ctx->fork_ev[d], r.st));
    for (cudaStream_t ss : ctx->side[d]) CUDA_TRY(cudaStreamWaitEvent(ss, ctx->fork_ev[d], 0));
  }
  size_t gi = 0;
  for (size_t i = 0; i < p.raw.size(); ++i) {
    const Group &g = p.raw[i];
    const uint32_t n = (uint32_t)g.order.size();
    const uint32_t *d_order = sh.d_order + g.order_off;
    const bool is_dom = r.events && (int)i == p.dom;
    cudaStream_t st = r.st;
    if (fan_out && !g.table_global && ((int)i != p.dom || g.mode == 3)) {
      const size_t k = g.mode == 3 ? 0 : 1 + gi++ % 2;
      st = ctx->side[d][k];
      r.side_used[k] = true;
    }
    print_plan(g);
    if (is_dom) CUDA_TRY(cudaEventRecord(ctx->ev[2], st));
    if (g.table_global) {
      const uint64_t slot_bytes = (uint64_t)g.lut_bytes + g.ent_bytes;
      // chunk: a multiple of 32 slots whose tables fit the scratch budget and 32-bit entry offsets
      uint64_t per = std::max<uint64_t>(32, std::min<uint64_t>(kTabArenaBudget / slot_bytes, 0xF0000000ull / slot_bytes) / 32 * 32);
      const uint64_t chunk = std::min<uint64_t>(per, align_up(n, 32));
      if (sh.tab_cap < chunk * slot_bytes) {
        cudaFree(sh.d_tab);
        sh.d_tab = nullptr;
        sh.tab_cap = 0;
        CUDA_TRY(cudaMalloc(&sh.d_tab, chunk * slot_bytes));
        sh.tab_cap = chunk * slot_bytes;
      }
      r.A.tab = sh.d_tab;
      for (uint64_t o = 0; o < n; o += chunk) {
        // tables in global memory: 32 lanes, the uniform LUT, the generic post-processing
        RansLaunch L = rans_launch(g, sh.d_streams, d_order + o, (uint32_t)std::min<uint64_t>(chunk, n - o), r.dump);
        L.lanes_per_warp = 32;
        L.lutb_bytes = 0;
        L.mode = 0;
        CUDA_TRY(dcb_launch_rans_raw(L, g.ncp, g.wide, true, r.A, st));
        r.stats.n_launches++;
      }
    } else {
      const RansLaunch L = rans_launch(g, sh.d_streams, d_order, n, r.dump);
      r.tl(st, g.mode == 1 ? "rans mode1" : g.mode == 2 ? "rans mode2" : g.mode == 3 ? "rans mode3" : g.mode == 4 ? "rans mode4" : "rans mode0");
      CUDA_TRY(g.rec_ka ? dcb_launch_rans_raw_rec(L, g.ncp, r.A, st)
               : g.pairs ? dcb_launch_rans_raw_pc(L, g.ncp, r.A, st) : dcb_launch_rans_raw(L, g.ncp, g.wide, false, r.A, st));
      r.tl(st);
      r.stats.n_launches++;
    }
    if (g.mode == 3) {
      // same stream, right behind the corrections; no shared memory, so they run next to the other groups' rANS kernels
      r.tl(st, "oct_chain");
      CUDA_TRY(dcb_launch_oct_chain(sh.d_streams, d_order, n, r.dump, r.A, st));
      r.tl(st);
      r.tl(st, "oct_unit");
      CUDA_TRY(dcb_launch_oct_unit(sh.d_streams, d_order, n, g.max_entries, r.A, st));
      r.tl(st);
      r.stats.n_launches += 2;
    }
    if (is_dom) {
      CUDA_TRY(cudaEventRecord(ctx->ev[3], st));
      ctx->ev_raw = true;
      note_dominant(r, g);
    }
    r.stats.n_streams += (int32_t)n;
  }
  return DCB_OK;
}

// Everything behind the rANS kernels: the flag kernels, the joins of the side streams, the post-processing, point-
// parallel and mesh prediction kernels, on the shard's stream.
int launch_after_rans(ShardRun &r, const ShardPlan &p, bool flags_early) {
  dcb_ctx *ctx = r.ctx;
  Shard &sh = r.sh;
  const int d = r.dev_index;
  const cudaStream_t st = r.st;
  const uint32_t dump = r.dump;
  DevArenas &A = r.A;
  dcb_launch_stats &stats = r.stats;
  auto launch_flag_kernels = [&](cudaStream_t fs, cudaStream_t gs) -> int {
    for (int n = 1; n <= 4; ++n)
      if (!p.cmp[n].order.empty()) {
        CUDA_TRY(dcb_launch_cmp_flags(sh.d_streams, sh.d_order + p.cmp[n].order_off, (uint32_t)p.cmp[n].order.size(), A, fs));
        stats.n_launches++;
      }
    if (!p.geo.order.empty()) {
      CUDA_TRY(dcb_launch_geo_flips(sh.d_streams, sh.d_order + p.geo.order_off, (uint32_t)p.geo.order.size(), A, gs));
      stats.n_launches++;
    }
    return DCB_OK;
  };
  if (flags_early) {  // issued behind the rANS launches so that those get their SMs first; crease flags and flip bits on a
    int rcf = launch_flag_kernels(ctx->side[d][2], ctx->side[d][1]);  // stream each (serial chains both)
    if (rcf) return rcf;
    r.side_used[2] = r.side_used[1] = true;
  }
  {  // mesh maps: behind the rANS launches (their chains hide the copy), in front of the parallelogram kernels
    int rcm = issue_maps_copy(ctx, r.b, sh, d);
    if (rcm) return rcm;
  }
  auto launch_cmp_deps = [&](cudaStream_t ds) -> int {
    for (int n = 1; n <= 4; ++n)
      if (!p.cmp[n].order.empty()) {
        CUDA_TRY(dcb_launch_cmp_deps(sh.d_streams, sh.d_order + p.cmp[n].order_off, (uint32_t)p.cmp[n].order.size(), p.cmp[n].max_entries, A, ds));
        stats.n_launches++;
      }
    return DCB_OK;
  };
  if (flags_early) {  // the dependency lists need the maps only: next to the rANS kernels as well, behind the maps' copy
    CUDA_TRY(cudaStreamWaitEvent(ctx->side[d][2], ctx->maps_ev[d], 0));
    int rcd = launch_cmp_deps(ctx->side[d][2]);
    if (rcd) return rcd;
  }
  for (int k = 0; k < 3; ++k)
    if (r.side_used[k]) {
      CUDA_TRY(cudaEventRecord(ctx->join_ev[d][k], ctx->side[d][k]));
      CUDA_TRY(cudaStreamWaitEvent(st, ctx->join_ev[d][k], 0));
    }
  if (!p.wide.order.empty()) {
    CUDA_TRY(dcb_launch_wide_post(sh.d_streams, sh.d_order + p.wide.order_off, (uint32_t)p.wide.order.size(), dump, A, st));
    stats.n_launches++;
  }
  for (int n = 1; n <= 4; ++n) {
    if (!p.post[n].order.empty()) {
      CUDA_TRY(dcb_launch_serial_post(sh.d_streams, sh.d_order + p.post[n].order_off, (uint32_t)p.post[n].order.size(), n, dump, 0, A, st));
      stats.n_launches++;
    }
    if (!p.par[n].order.empty()) {
      const ShardPlan::ParPost &pp = p.pp[n];
      const uint32_t np = (uint32_t)p.par[n].order.size();
      const bool time_par = r.events && !ctx->ev_par;
      if (time_par) {
        CUDA_TRY(cudaEventRecord(ctx->ev[6], st));
        for (uint32_t si : p.par[n].order) {
          const StreamDesc &sd = sh.streams[si];
          ctx->algo_par += sd.out_bytes + (sd.scheme == SCHEME_TAGGED ? sd.n_entries
                                                                       : (uint64_t)sd.n_entries * sd.ncp * sd.raw_num_bytes);
          if (sd.scheme == SCHEME_TAGGED) ctx->par_streams.push_back({&sh, si});  // + its bit area, once bits_total is back
        }
      }
      uint32_t *d_runs = sh.d_order + pp.runs_off;
      const uint32_t n_prefix = pp.rounds ? pp.rounds : np;  // entries of the run prefix (rounds or streams)
      CUDA_TRY(dcb_launch_par_post(sh.d_streams, sh.d_order + p.par[n].order_off, d_runs, np, pp.runs[n_prefix], pp.run_len,
                                   pp.claim, pp.rounds, d_runs + n_prefix + 1, r.num_sms, n, dump, next_epoch(sh), A, st));
      stats.n_launches += 1;
      if (pp.delta) {
        // streams whose corrections break the modular-sum condition fall back to the exact serial recurrence
        CUDA_TRY(dcb_launch_serial_post(sh.d_streams, sh.d_order + p.par[n].order_off, np, n, dump, 1, A, st));
        stats.n_launches++;
      }
      if (time_par) {
        CUDA_TRY(cudaEventRecord(ctx->ev[7], st));
        ctx->ev_par = true;
      }
    }
  }
  if (!p.octc.order.empty()) {  // octahedral recurrence of the normals whose corrections par_post2 left in the scratch
    CUDA_TRY(dcb_launch_oct_chain(sh.d_streams, sh.d_order + p.octc.order_off, (uint32_t)p.octc.order.size(), dump, A, st));
    stats.n_launches++;
  }
  if (!p.octs.order.empty()) {
    CUDA_TRY(dcb_launch_oct_unit(sh.d_streams, sh.d_order + p.octs.order_off, (uint32_t)p.octs.order.size(), p.octs.max_entries, A, st));
    stats.n_launches++;
  }
  if (!p.copy.order.empty()) {
    CUDA_TRY(dcb_launch_copy(sh.d_streams, sh.d_order + p.copy.order_off, (uint32_t)p.copy.order.size(), p.copy.max_bytes, A, st));
    stats.n_launches++;
  }
  // mesh prediction stage (ms_para of the stats): parallelogram, constrained multi-parallelogram, tex-coord and
  // geometric-normal kernels, timed as one span
  bool any_mesh_stage = !p.tex.order.empty() || !p.geo.order.empty();
  for (int n = 1; n <= 4; ++n) any_mesh_stage = any_mesh_stage || !p.para[n].order.empty() || !p.cmp[n].order.empty();
  const bool time_para = r.events && !ctx->ev_para && any_mesh_stage;
  if (time_para) CUDA_TRY(cudaEventRecord(ctx->ev[8], st));
  for (int n = 1; n <= 4; ++n)
    if (!p.para[n].order.empty()) {
      CUDA_TRY(dcb_launch_para(sh.d_streams, sh.d_order + p.para[n].order_off, (uint32_t)p.para[n].order.size(), n,
                               p.para[n].max_entries, dump, A, st));
      stats.n_launches += 2;
    }
  if (p.flag_kernels() && !flags_early) {
    int rcf = launch_flag_kernels(st, st);
    if (rcf) return rcf;
    rcf = launch_cmp_deps(st);
    if (rcf) return rcf;
  }
  for (int n = 1; n <= 4; ++n)
    if (!p.cmp[n].order.empty()) {  // constrained multi-parallelogram: the chain
      CUDA_TRY(dcb_launch_cmp(sh.d_streams, sh.d_order + p.cmp[n].order_off, (uint32_t)p.cmp[n].order.size(), n, dump, A, st));
      stats.n_launches++;
    }
  if (!p.tex.order.empty()) {  // behind the parallelogram kernels: the predictor reads the decoded positions of its parent
    CUDA_TRY(dcb_launch_tex(sh.d_streams, sh.d_order + p.tex.order_off, (uint32_t)p.tex.order.size(), p.tex.max_entries, dump, A, st));
    stats.n_launches += 2;
  }
  if (!p.geo.order.empty()) {  // behind the parallelogram kernels: the predictor reads the decoded positions of its parent
    CUDA_TRY(dcb_launch_geo_normal(sh.d_streams, sh.d_order + p.geo.order_off, (uint32_t)p.geo.order.size(), p.geo.max_entries, dump, A, st));
    stats.n_launches++;
  }
  if (time_para) {
    CUDA_TRY(cudaEventRecord(ctx->ev[9], st));
    ctx->ev_para = true;
  }
  return DCB_OK;
}

// Decode everything of one shard into (d_out, d_dbg).  Asynchronous on the shard's stream except
// for the resolve round trips of Tagged streams.
int decode_shard(dcb_ctx *ctx, dcb_batch *b, Shard &sh, int dev_index, uint8_t *d_out, uint8_t *d_dbg, uint32_t flags,
                 bool timed) {
  cudaStream_t st = ctx->streams[dev_index];
  CUDA_TRY(cudaSetDevice(sh.device));
  const uint32_t num_sms = (uint32_t)ctx->num_sms[dev_index];
  // device 0 of the context writes the decode's statistics record; the other devices' decode threads count their
  // launches and streams in records of their own, merged by finish_stats
  dcb_launch_stats &stats = dev_index == 0 ? ctx->stats : ctx->dev_stats[dev_index];
  if (sh.streams.empty()) return DCB_OK;
  int rc = reset_descriptors(sh, st);
  if (rc) return rc;
  // point order: the kernels write the entry-order staging, the point stage fills d_out from it
  ShardRun r{ctx, b, sh, dev_index, st, num_sms, stats, DevArenas{sh.d_in, sh.pts ? sh.d_pts : d_out, d_dbg, sh.d_aux, sh.d_tab, sh.d_maps},
             flags & (DCB_DUMP_SYMBOLS | DCB_DUMP_QINTS), timed && dev_index == 0,
             timed && sh.device == ctx->devices[0] && env_flags().debug_timing};
  if (r.events) CUDA_TRY(cudaEventRecord(ctx->ev[0], st));
  bool deferred_descs = false;
  if ((rc = run_tag_rounds(r, deferred_descs))) return rc;
  ShardPlan &p = sh.plan;
  if ((rc = plan_shard(b, sh, num_sms, p))) return rc;
  if (!p.order.empty()) {
    if ((rc = ensure_order(sh, p.order.size()))) return rc;
    CUDA_TRY(cudaMemcpyAsync(sh.d_order, p.order.data(), p.order.size() * 4, cudaMemcpyHostToDevice, st));
    // crease flags / flip bits of the 8f-3 predictors depend on the bitstream only: their (serial, small) rABS kernels
    // run on a side stream next to the rANS kernels -- unless descriptors are still being resolved on the device behind
    // Tagged bit areas
    const bool flags_early = p.flag_kernels() && !deferred_descs;
    if ((rc = launch_rans_groups(r, p, flags_early))) return rc;
    if ((rc = launch_after_rans(r, p, flags_early))) return rc;
  }
  if (sh.pts) {  // last writer of every attribute: behind the joins, on the main stream
    if ((rc = issue_maps_copy(ctx, b, sh, dev_index))) return rc;
    DevArenas P = r.A;
    P.out = d_out;
    r.tl(st, "point stage");
    CUDA_TRY(dcb_launch_point_stage(sh.pstage, sh.d_streams, P, num_sms, st));
    r.tl(st);
    stats.n_launches += 3;
  }
  if (r.events) CUDA_TRY(cudaEventRecord(ctx->ev[1], st));
  // parallelogram kernels and the point stage validate the caller's maps on the device, resumed walks parse and
  // validate on the device: their verdicts travel back behind the kernels and are folded in after the caller's
  // synchronisation
  if (p.has_para || deferred_descs || sh.pts) return queue_desc_copyback(ctx, sh, st);
  return DCB_OK;
}

// after a decode: fold walk / stream statuses into the buffer records
void collect_status(dcb_batch *b) {
  absorb_descs(b);
  for (BufRec &r : b->bufs) {
    if (r.info.status) continue;
    const Shard &sh = b->shards[r.shard];
    const BufWalk &w = sh.walks[r.local];
    if (w.status) { r.info.status = w.status; continue; }
    for (int i = 0; i < w.stream_count; ++i) {
      const StreamDesc &s = sh.streams[w.stream_first + i];
      if (s.status) { r.info.status = s.status; break; }
    }
    if (!r.info.status && r.idx_job >= 0 && sh.h_fstatus) r.info.status = sh.h_fstatus[r.idx_job];
  }
}

void tl_mark(dcb_ctx *ctx, const std::string &name, cudaStream_t s, bool begin) {
  if (!env_flags().debug_timing) return;
  if (begin) {
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, s);
    ctx->timeline.push_back({name, {a, b}});
  } else {
    cudaEventRecord(ctx->timeline.back().second.second, s);
  }
}

// D2H of one shard's arenas (asynchronous).  Pipeline slices: in slice order on the device's download stream.
int download_shard(dcb_ctx *ctx, dcb_batch *b, int d, uint8_t *host_out, uint8_t *host_dbg) {
  Shard &sh = b->shards[d];
  CUDA_TRY(cudaSetDevice(sh.device));
  if (host_out && sh.ext_out && sh.out_bytes) {
    if (sh.share > 1) {  // the slice's own stream then waits for the copy, so that sync_all covers it
      cudaStream_t cs = ctx->copy_out[d];
      CUDA_TRY(cudaEventRecord(ctx->out_ev[d], ctx->streams[d]));
      CUDA_TRY(cudaStreamWaitEvent(cs, ctx->out_ev[d], 0));
      tl_mark(ctx, "d2h s" + std::to_string(d), cs, true);
      CUDA_TRY(cudaMemcpyAsync(host_out + sh.out_base, sh.ext_out, sh.out_bytes, cudaMemcpyDeviceToHost, cs));
      tl_mark(ctx, "", cs, false);
      CUDA_TRY(cudaEventRecord(ctx->out_ev[d], cs));
      CUDA_TRY(cudaStreamWaitEvent(ctx->streams[d], ctx->out_ev[d], 0));
    } else {
      CUDA_TRY(cudaMemcpyAsync(host_out + sh.out_base, sh.ext_out, sh.out_bytes, cudaMemcpyDeviceToHost, ctx->streams[d]));
    }
  }
  if (host_dbg && sh.ext_dbg && sh.dbg_bytes)
    CUDA_TRY(cudaMemcpyAsync(host_dbg + sh.dbg_base, sh.ext_dbg, sh.dbg_bytes, cudaMemcpyDeviceToHost, ctx->streams[d]));
  return DCB_OK;
}

int sync_all(dcb_ctx *ctx);
int decode_all_impl(dcb_ctx *ctx, dcb_batch *b, void *dev_out, void *dev_dbg, uint32_t flags, uint8_t *host_out, uint8_t *host_dbg);

// An error in the middle of a batch must not leave kernels or copies of the shards launched so far in flight: the
// caller frees the batch next, and its arenas go back to the context's cache.
void drain(dcb_ctx *ctx) {
  (void)sync_all(ctx);
  for (size_t d = 0; d < ctx->devices.size(); ++d) {  // side and copy streams too
    cudaSetDevice(ctx->devices[d]);
    cudaDeviceSynchronize();
  }
  cudaGetLastError();
}

int decode_all(dcb_ctx *ctx, dcb_batch *b, void *dev_out, void *dev_dbg, uint32_t flags, uint8_t *host_out = nullptr,
               uint8_t *host_dbg = nullptr) {
  const int rc = decode_all_impl(ctx, b, dev_out, dev_dbg, flags, host_out, host_dbg);
  if (rc != DCB_OK && ctx) drain(ctx);
  return rc;
}

int decode_all_impl(dcb_ctx *ctx, dcb_batch *b, void *dev_out, void *dev_dbg, uint32_t flags, uint8_t *host_out,
                    uint8_t *host_dbg) {
  if (!ctx || !b) return DCB_ERR_ARG;
  if ((int)ctx->devices.size() != b->n_devices) return DCB_ERR_ARG;
  if ((dev_out || dev_dbg) && b->n_devices != 1) return DCB_ERR_ARG;
  const uint32_t dump = flags & (DCB_DUMP_SYMBOLS | DCB_DUMP_QINTS);
  if (dump == (DCB_DUMP_SYMBOLS | DCB_DUMP_QINTS)) return DCB_ERR_ARG;  // one debug arena
  for (const BufRec &r : b->bufs)
    if (r.info.needs_connectivity && r.info.status == DCB_OK) return DCB_ERR_STATE;  // dcb_index_finish not run
  memset(&ctx->stats, 0, sizeof ctx->stats);
  ctx->dev_stats.assign(ctx->devices.size(), dcb_launch_stats{});
  ctx->par_streams.clear();
  ctx->ev_raw = ctx->ev_tag = ctx->ev_par = ctx->ev_para = false;
  ctx->algo_raw = ctx->algo_tag = ctx->algo_par = 0;
  ctx->raw_name[0] = 0;
  const auto t_up = std::chrono::steady_clock::now();
  for (int d = 0; d < b->n_devices; ++d) {
    Shard &sh = b->shards[d];
    int rc = upload_shard(ctx, b, sh, d);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(sh.device));
    uint8_t *o = (uint8_t *)dev_out;
    if (!o) {
      if (!sh.d_out && sh.out_bytes) {
        CUDA_TRY(pool_alloc(sh.pool, sh.device, sh.out_bytes, &sh.d_out, &sh.cap_out));
        sh.own_out = true;
      }
      o = sh.d_out;
    }
    sh.ext_out = o;
    uint8_t *g = (uint8_t *)dev_dbg;
    if (dump && !g) {
      if (sh.dbg_cap < sh.dbg_bytes) {
        cudaFree(sh.d_dbg);
        sh.d_dbg = nullptr;
        sh.dbg_cap = 0;
        CUDA_TRY(cudaMalloc(&sh.d_dbg, std::max<uint64_t>(sh.dbg_bytes, 16)));
        sh.dbg_cap = std::max<uint64_t>(sh.dbg_bytes, 16);
      }
      g = sh.d_dbg;
    }
    sh.ext_dbg = g;
  }
  const bool dbg_t = env_flags().debug_timing;
  if (dbg_t)
    fprintf(stderr, "[dcb timing] uploads issued in %.1f ms\n",
            std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_up).count());
  const auto t0 = std::chrono::steady_clock::now();
  auto run_shard = [&](int d) -> int {
    Shard &sh = b->shards[d];
    int rc = issue_arena_copy(ctx, b, sh, d);
    if (rc) return rc;
    rc = decode_shard(ctx, b, sh, d, sh.ext_out, sh.ext_dbg, flags, true);
    if (rc) return rc;
    rc = faces_shard(ctx, b, sh, d, sh.ext_out);
    if (rc) return rc;
    if (host_out || host_dbg) {  // host-buffer decode: this shard's results start travelling while the next one decodes
      rc = download_shard(ctx, b, d, host_out, host_dbg);
      if (rc) return rc;
    }
    if (dbg_t)
      fprintf(stderr, "[dcb timing]   shard %d launched at +%.1f ms (direct=%d in=%.1f MB out=%.1f MB)\n", d,
              std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(), (int)sh.direct,
              sh.in_bytes / 1e6, sh.out_bytes / 1e6);
    return DCB_OK;
  };
  // One host thread per PHYSICAL device (SURVEY 8e): a shard whose decode needs a round trip (a Tagged attribute followed
  // by more attributes) holds only its own device's thread.  Pipeline slices of one device stay on one thread, in slice
  // order -- their bulk copies share one stream per direction.
  std::vector<std::vector<int>> by_dev;
  {
    std::vector<int> ids;
    for (int d = 0; d < b->n_devices; ++d) {
      size_t k = 0;
      while (k < ids.size() && ids[k] != b->shards[d].device) ++k;
      if (k == ids.size()) { ids.push_back(b->shards[d].device); by_dev.emplace_back(); }
      by_dev[k].push_back(d);
    }
  }
  if (by_dev.size() <= 1 || dbg_t || env_flags().no_threads) {
    for (int d = 0; d < b->n_devices; ++d) {
      int rc = run_shard(d);
      if (rc) return rc;
    }
    return DCB_OK;
  }
  std::vector<int> rcs(by_dev.size(), DCB_OK);
  std::vector<std::thread> workers;
  for (size_t k = 1; k < by_dev.size(); ++k)
    workers.emplace_back([&, k]() {
      for (int d : by_dev[k]) {
        try {
          rcs[k] = run_shard(d);
        } catch (const std::bad_alloc &) {
          rcs[k] = DCB_ERR_OOM;
        } catch (...) {
          rcs[k] = DCB_ERR_STATE;
        }
        if (rcs[k]) break;
      }
    });
  for (int d : by_dev[0]) {
    rcs[0] = run_shard(d);
    if (rcs[0]) break;
  }
  for (std::thread &t : workers) t.join();
  for (int rc : rcs)
    if (rc) return rc;
  return DCB_OK;
}

int sync_all(dcb_ctx *ctx) {
  for (size_t d = 0; d < ctx->devices.size(); ++d) {
    CUDA_TRY(cudaSetDevice(ctx->devices[d]));
    CUDA_TRY(cudaStreamSynchronize(ctx->streams[d]));
  }
  return DCB_OK;
}

void finish_stats(dcb_ctx *ctx) {
  dcb_launch_stats &st = ctx->stats;
  for (size_t d = 1; d < ctx->dev_stats.size(); ++d) {
    st.n_launches += ctx->dev_stats[d].n_launches;
    st.n_streams += ctx->dev_stats[d].n_streams;
  }
  for (auto &ps : ctx->par_streams)
    ctx->algo_par += (static_cast<const Shard *>(ps.first)->streams[ps.second].bits_total + 7) / 8;
  ctx->par_streams.clear();
  float ms = 0.0f;
  for (auto &t : ctx->timeline) {
    float a = 0.0f, b = 0.0f;
    cudaEventElapsedTime(&a, ctx->ev[0], t.second.first);
    cudaEventElapsedTime(&b, ctx->ev[0], t.second.second);
    fprintf(stderr, "[dcb timeline] %-12s %8.2f -> %8.2f ms\n", t.first.c_str(), a, b);
    cudaEventDestroy(t.second.first);
    cudaEventDestroy(t.second.second);
  }
  ctx->timeline.clear();
  if (cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]) == cudaSuccess) st.ms_total = ms;
  else cudaGetLastError();
  if (ctx->ev_raw && cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]) == cudaSuccess) st.ms_raw = ms;
  if (ctx->ev_tag && cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]) == cudaSuccess) st.ms_tag = ms;
  if (ctx->ev_par && cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7]) == cudaSuccess) st.ms_par = ms;
  if (ctx->ev_para && cudaEventElapsedTime(&ms, ctx->ev[8], ctx->ev[9]) == cudaSuccess) st.ms_para = ms;
  cudaGetLastError();
  if (st.ms_raw >= st.ms_tag && st.ms_raw >= st.ms_par && ctx->ev_raw) {
    st.ms_dominant = st.ms_raw;
    st.algo_bytes_dominant = ctx->algo_raw;
    snprintf(st.dominant_name, sizeof st.dominant_name, "%s", ctx->raw_name);
  } else if (st.ms_tag >= st.ms_par && ctx->ev_tag) {
    st.ms_dominant = st.ms_tag;
    st.algo_bytes_dominant = ctx->algo_tag;
    snprintf(st.dominant_name, sizeof st.dominant_name, "rans_tag_kernel (tag stream of the Tagged scheme)");
  } else if (ctx->ev_par) {
    st.ms_dominant = st.ms_par;
    st.algo_bytes_dominant = ctx->algo_par;
    snprintf(st.dominant_name, sizeof st.dominant_name, "par_post_kernel passes (bit extract + scan + store)");
  }
}

}  // namespace

// No C++ exception crosses the C ABI: every entry point that can allocate runs inside this barrier.
template <typename F>
static int guarded(F &&f) {
  try {
    return f();
  } catch (const std::bad_alloc &) {
    return DCB_ERR_OOM;
  } catch (...) {
    return DCB_ERR_STATE;
  }
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int dcb_version(void) { return DCB_VERSION; }

int dcb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
  }
  return ok;
}

const char *dcb_error_string(int code) {
  switch (code) {
    case DCB_OK: return "ok";
    case DCB_ERR_EOF: return "unexpected end of buffer";
    case DCB_ERR_MAGIC: return "not a Draco buffer";
    case DCB_ERR_UNSUPPORTED: return "unsupported bitstream feature";
    case DCB_ERR_SCHEME: return "invalid symbol coding scheme";
    case DCB_ERR_BITLEN: return "invalid symbol bit length";
    case DCB_ERR_TABLE: return "invalid rANS probability table";
    case DCB_ERR_RANS_INIT: return "invalid rANS stream";
    case DCB_ERR_PRED: return "invalid prediction scheme";
    case DCB_ERR_WRAP: return "invalid wrap transform bounds";
    case DCB_ERR_QUANT: return "invalid quantization parameters";
    case DCB_ERR_ATTR: return "invalid attribute descriptor";
    case DCB_ERR_TAG: return "invalid tagged bit length";
    case DCB_ERR_NUM_SYMBOLS: return "empty symbol alphabet";
    case DCB_ERR_MAPS: return "missing or inconsistent mesh connectivity maps";
    case DCB_ERR_CONNECTIVITY: return "connectivity decode failed";
    case DCB_ERR_ARG: return "invalid argument";
    case DCB_ERR_NO_DEVICE: return "no sm_100 CUDA device (there is no CPU fallback)";
    case DCB_ERR_CUDA: return "CUDA error";
    case DCB_ERR_OOM: return "out of memory";
    case DCB_ERR_STATE: return "call order violated";
    default: return "unknown error";
  }
}

int dcb_create(const int *device_ids, int n_devices, dcb_ctx **out) {
  return guarded([&]() -> int {
    if (!out || n_devices < 0) return DCB_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
      cudaGetLastError();
      return DCB_ERR_NO_DEVICE;
    }
    dcb_ctx *c = new (std::nothrow) dcb_ctx();
    if (!c) return DCB_ERR_OOM;
    if (!device_ids || n_devices == 0) {
      int cur = 0;
      if (cudaGetDevice(&cur) != cudaSuccess) { delete c; return DCB_ERR_NO_DEVICE; }
      c->devices.push_back(cur);
    } else {
      for (int i = 0; i < n_devices; ++i) c->devices.push_back(device_ids[i]);
    }
    for (int dev : c->devices) {
      cudaDeviceProp p;
      if (dev < 0 || dev >= count || cudaGetDeviceProperties(&p, dev) != cudaSuccess || p.major != 10) {
        cudaGetLastError();
        dcb_destroy(c);
        return DCB_ERR_NO_DEVICE;  // kernels are sm_100a only: no fallback
      }
      cudaStream_t st = nullptr;
      if (cudaSetDevice(dev) != cudaSuccess || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
        cudaGetLastError();
        dcb_destroy(c);
        return DCB_ERR_CUDA;
      }
      c->streams.push_back(st);
      c->own_stream.push_back(true);
      std::vector<cudaStream_t> side(3, nullptr);
      std::vector<cudaEvent_t> jev(3, nullptr);
      cudaEvent_t fev = nullptr;
      // side[0] outranks the others: it carries the group whose chain goes on after its rANS kernel (normals:
      // oct_chain, oct_unit), the longest dependent sequence of a batch
      int prio_lo = 0, prio_hi = 0;
      cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
      for (int k = 0; k < 3; ++k) {
        if (k == 0) cudaStreamCreateWithPriority(&side[k], cudaStreamNonBlocking, prio_hi);
        else cudaStreamCreateWithFlags(&side[k], cudaStreamNonBlocking);
        cudaEventCreateWithFlags(&jev[k], cudaEventDisableTiming);
      }
      cudaEventCreateWithFlags(&fev, cudaEventDisableTiming);
      c->side.push_back(side);
      c->join_ev.push_back(jev);
      c->fork_ev.push_back(fev);
      {
        cudaStream_t ci = nullptr, co = nullptr;
        bool own = true;
        for (size_t e = 0; e + 1 < c->streams.size(); ++e)
          if (c->devices[e] == dev) { ci = c->copy_in[e]; co = c->copy_out[e]; own = false; break; }
        if (own) {
          cudaStreamCreateWithFlags(&ci, cudaStreamNonBlocking);
          cudaStreamCreateWithFlags(&co, cudaStreamNonBlocking);
        }
        c->copy_in.push_back(ci);
        c->copy_out.push_back(co);
        c->own_copy.push_back(own);
        cudaEvent_t ie = nullptr, oe = nullptr, me = nullptr;
        cudaEventCreateWithFlags(&ie, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&oe, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&me, cudaEventDisableTiming);
        c->in_ev.push_back(ie);
        c->out_ev.push_back(oe);
        c->maps_ev.push_back(me);
      }
      c->num_sms.push_back(p.multiProcessorCount > 0 ? p.multiProcessorCount : (int)kNumSMsDefault);
    }
    cudaSetDevice(c->devices[0]);
    for (auto &e : c->ev) cudaEventCreate(&e);
    *out = c;
    return DCB_OK;
  });
}

void dcb_destroy(dcb_ctx *ctx) {
  if (!ctx) return;
  pool_trim(ctx->pool);
  ctx->pool->cached = kPoolCap + 1;  // batches freed after their context: straight to cudaFree
  for (size_t i = 0; i < ctx->streams.size(); ++i)
    if (ctx->own_stream[i]) {
      cudaSetDevice(ctx->devices[i]);
      cudaStreamDestroy(ctx->streams[i]);
    }
  for (auto &e : ctx->ev)
    if (e) cudaEventDestroy(e);
  for (size_t i = 0; i < ctx->side.size(); ++i) {
    cudaSetDevice(ctx->devices[i]);
    for (auto &s : ctx->side[i]) if (s) cudaStreamDestroy(s);
    for (auto &e : ctx->join_ev[i]) if (e) cudaEventDestroy(e);
    if (ctx->fork_ev[i]) cudaEventDestroy(ctx->fork_ev[i]);
    if (i < ctx->own_copy.size() && ctx->own_copy[i]) {
      if (ctx->copy_in[i]) cudaStreamDestroy(ctx->copy_in[i]);
      if (ctx->copy_out[i]) cudaStreamDestroy(ctx->copy_out[i]);
    }
    if (i < ctx->in_ev.size() && ctx->in_ev[i]) cudaEventDestroy(ctx->in_ev[i]);
    if (i < ctx->out_ev.size() && ctx->out_ev[i]) cudaEventDestroy(ctx->out_ev[i]);
    if (i < ctx->maps_ev.size() && ctx->maps_ev[i]) cudaEventDestroy(ctx->maps_ev[i]);
  }
  delete ctx;
}

int dcb_set_stream(dcb_ctx *ctx, int dev_index, void *cuda_stream) {
  return guarded([&]() -> int {
    if (!ctx || dev_index < 0 || dev_index >= (int)ctx->streams.size()) return DCB_ERR_ARG;
    if (ctx->own_stream[dev_index]) {
      cudaSetDevice(ctx->devices[dev_index]);
      cudaStreamDestroy(ctx->streams[dev_index]);
    }
    ctx->streams[dev_index] = (cudaStream_t)cuda_stream;
    ctx->own_stream[dev_index] = false;
    return DCB_OK;
  });
}

int dcb_set_limits(dcb_ctx *ctx, uint64_t max_points_per_buffer, uint64_t points_per_byte) {
  if (!ctx) return DCB_ERR_ARG;
  ctx->max_points = max_points_per_buffer;
  ctx->points_per_byte = points_per_byte;
  return DCB_OK;
}

int dcb_index(dcb_ctx *ctx, const uint8_t *const *bufs, const uint64_t *lens, int n_bufs, dcb_batch **out) {
  return guarded([&]() -> int {
    int rc = make_batch(ctx, nullptr, bufs, nullptr, lens, n_bufs, out);
    if (rc == DCB_OK) finalize_layout(*out);
    return rc;
  });
}

int dcb_index_arena(dcb_ctx *ctx, const uint8_t *arena, const uint64_t *offs, const uint64_t *lens, int n_bufs,
                    dcb_batch **out) {
  return guarded([&]() -> int {
    if (!arena || !offs) return DCB_ERR_ARG;
    int rc = make_batch(ctx, arena, nullptr, offs, lens, n_bufs, out);
    if (rc == DCB_OK) finalize_layout(*out);
    return rc;
  });
}

int dcb_get_buffer_info(const dcb_batch *b, int buf, dcb_buffer_info *out) {
  return guarded([&]() -> int {
    if (!b || !out || buf < 0 || buf >= (int)b->bufs.size()) return DCB_ERR_ARG;
    *out = b->bufs[buf].info;
    return DCB_OK;
  });
}

int dcb_get_attr_info(const dcb_batch *b, int buf, int attr, dcb_attr_info *out) {
  return guarded([&]() -> int {
    if (!b || !out || buf < 0 || buf >= (int)b->bufs.size()) return DCB_ERR_ARG;
    const BufRec &r = b->bufs[buf];
    const Shard &sh = b->shards[r.shard];
    const BufWalk &w = sh.walks[r.local];
    if (attr < 0 || attr >= w.stream_count) return DCB_ERR_ARG;
    const StreamDesc &s = sh.streams[w.stream_first + attr];
    memset(out, 0, sizeof *out);
    out->att_type = s.att_type;
    out->data_type = s.data_type;
    out->num_components = s.nc;
    out->normalized = s.normalized;
    out->unique_id = s.unique_id;
    out->seq_decoder_type = s.seq_type;
    out->decoder_id = s.decoder_id;
    out->pred_method = s.pred_method;
    out->transform = s.transform;
    out->scheme = (s.scheme == SCHEME_TAGGED || s.scheme == SCHEME_RAW) ? (int32_t)s.scheme : -1;
    out->precision_bits = s.prec_bits;
    out->n_entries = s.n_entries;
    out->out_bytes = sh.fin_bytes[w.stream_first + attr];
    out->out_off = sh.out_base + sh.fin_off[w.stream_first + attr];
    out->dbg_off = sh.dbg_base + s.dbg_off;
    out->xf_a = s.xf_a;
    out->xf_b = s.xf_b;
    for (int c = 0; c < 4; ++c) out->q_min[c] = s.q_min[c];
    out->q_range = s.q_range;
    out->q_bits = s.q_bits;
    out->resolved = s.state == ST_READY;
    return DCB_OK;
  });
}

uint64_t dcb_batch_out_bytes(const dcb_batch *b) { return b ? b->total_out : 0; }
uint64_t dcb_batch_dbg_bytes(const dcb_batch *b) { return b ? b->total_dbg : 0; }
uint64_t dcb_batch_in_bytes(const dcb_batch *b) { return b ? b->total_in : 0; }
uint64_t dcb_batch_points(const dcb_batch *b) { return b ? b->total_points : 0; }
uint64_t dcb_batch_algo_bytes(const dcb_batch *b) { return b ? b->algo_bytes : 0; }

int dcb_set_attr_section(dcb_batch *b, int buf, uint64_t attr_section_off, uint32_t n_points) {
  return guarded([&]() -> int {
    if (!b || buf < 0 || buf >= (int)b->bufs.size()) return DCB_ERR_ARG;
    BufRec &r = b->bufs[buf];
    if (!r.info.needs_connectivity) return DCB_ERR_STATE;
    if (attr_section_off > r.len) return DCB_ERR_ARG;
    r.info.attr_section_off = attr_section_off;
    r.info.n_points = n_points;
    return DCB_OK;
  });
}

int dcb_set_mesh_maps(dcb_batch *b, int buf, int attr_decoder, const uint32_t *opposite,
                      const uint32_t *corner_to_vertex, uint64_t n_corners, const uint32_t *data_to_corner,
                      uint64_t n_entries, const int32_t *vertex_to_data, uint64_t n_vertices) {
  return guarded([&]() -> int {
    if (!b || buf < 0 || buf >= (int)b->bufs.size() || attr_decoder < 0 || attr_decoder > 255) return DCB_ERR_ARG;
    if ((n_corners && (!opposite || !corner_to_vertex)) || (n_entries && !data_to_corner) || (n_vertices && !vertex_to_data))
      return DCB_ERR_ARG;
    if (n_corners > 0xFFFFFFFFull || n_entries > 0xFFFFFFFFull || n_vertices > 0xFFFFFFFFull) return DCB_ERR_ARG;
    BufRec &r = b->bufs[buf];
    if (!r.info.needs_connectivity) return DCB_ERR_STATE;
    if (n_corners % 3 != 0) return DCB_ERR_ARG;  // corners come in triangles (CornerTable.Next / Previous)
    if (r.maps.size() <= (size_t)attr_decoder) r.maps.resize((size_t)attr_decoder + 1);
    MeshMapsHost &m = r.maps[attr_decoder];
    m.own.reset();
    m.opposite = opposite;
    m.corner_to_vertex = corner_to_vertex;
    m.data_to_corner = data_to_corner;
    m.vertex_to_data = vertex_to_data;
    m.n_corners = n_corners;
    m.n_entries = n_entries;
    m.n_vertices = n_vertices;
    m.set = true;
    return DCB_OK;
  });
}

int dcb_host_connectivity(dcb_batch *b, int buf) {
  return guarded([&]() -> int {
    if (!b || buf < 0 || buf >= (int)b->bufs.size()) return DCB_ERR_ARG;
    BufRec &r = b->bufs[buf];
    if (!r.info.needs_connectivity) return DCB_ERR_STATE;
    if (r.info.status != DCB_OK) return DCB_OK;
    if (!r.is_eb) {  // sequential mesh connectivity (MeshSequentialDecoder.cs:8-118, SURVEY 8f-4): indices on the host,
                     // attributes through the sequential (point-cloud) kernels -- no maps
      uint64_t attr_off = 0;
      uint32_t n_points = 0;
      int st;
      try {
        // DCB_FACES_ARENA: plain indices are located, the GPU decodes them into the arena
        r.seq_loc = DcbSeqIndexLoc{};
        r.faces.clear();
        st = dcb_host_sequential(r.src, r.len, r.conn_off, &attr_off, &n_points, &r.faces,
                                 b->faces == DCB_FACES_ARENA ? &r.seq_loc : nullptr);
      } catch (const std::bad_alloc &) {
        st = DCB_ERR_OOM;
      } catch (...) {
        st = DCB_ERR_CONNECTIVITY;
      }
      if (st != DCB_OK) {
        r.info.status = st;
        return DCB_OK;
      }
      r.info.attr_section_off = attr_off;
      r.info.n_points = n_points;
      r.pt_faces_set = true;  // faces for DCB_FACES_ARENA: decoded here, or located for the GPU
      r.pt_faces = r.faces.empty() ? nullptr : r.faces.data();
      r.pt_n_faces = r.faces.size() / 3;
      return DCB_OK;
    }
    std::vector<DcbHostMaps> maps;
    uint64_t attr_off = 0;
    uint32_t n_points = 0;
    int st;
    try {
      st = dcb_host_edgebreaker(r.src, r.len, r.conn_off, &attr_off, &n_points, &maps, &r.faces);
    } catch (const std::bad_alloc &) {  // counts the data cannot back: this buffer only
      st = DCB_ERR_OOM;
    } catch (...) {
      st = DCB_ERR_CONNECTIVITY;
    }
    if (st != DCB_OK) {  // the buffer fails alone, like an exception in the reference's DecodeConnectivity
      r.info.status = st;
      return DCB_OK;
    }
    r.info.attr_section_off = attr_off;
    r.info.n_points = n_points;
    r.maps.assign(maps.size(), MeshMapsHost{});
    for (size_t d = 0; d < maps.size(); ++d) {
      MeshMapsHost &m = r.maps[d];
      m.own = std::make_shared<DcbHostMaps>();
      m.own->opposite.swap(maps[d].opposite);
      m.own->corner_to_vertex.swap(maps[d].corner_to_vertex);
      m.own->data_to_corner.swap(maps[d].data_to_corner);
      m.own->vertex_to_data.swap(maps[d].vertex_to_data);
      m.opposite = m.own->opposite.data();
      m.corner_to_vertex = m.own->corner_to_vertex.data();
      m.data_to_corner = m.own->data_to_corner.data();
      m.vertex_to_data = m.own->vertex_to_data.data();
      m.n_corners = m.own->opposite.size();
      m.n_entries = m.own->data_to_corner.size();
      m.n_vertices = m.own->vertex_to_data.size();
      m.set = true;
    }
    // point order: the faces just decoded; when they are the corner table of decoder 0 (no attribute seams:
    // AssignPointsToCorners without attribute data) the NULL form gives the same map and uploads nothing
    r.pt_faces_set = true;
    r.pt_faces = nullptr;
    r.pt_n_faces = 0;
    if (r.maps.empty() || r.maps[0].n_corners != r.faces.size() ||
        memcmp(r.maps[0].corner_to_vertex, r.faces.data(), r.faces.size() * 4) != 0) {
      r.pt_faces = r.faces.data();
      r.pt_n_faces = r.faces.size() / 3;
    }
    return DCB_OK;
  });
}

int dcb_mesh_faces(const dcb_batch *b, int buf, uint32_t *faces, uint64_t cap_faces, uint64_t *n_faces) {
  return guarded([&]() -> int {
    if (!b || buf < 0 || buf >= (int)b->bufs.size() || !n_faces) return DCB_ERR_ARG;
    const BufRec &r = b->bufs[buf];
    if (r.seq_loc.located) return DCB_ERR_STATE;  // decoded on the GPU, into the output arena
    *n_faces = r.faces.size() / 3;
    if (faces) {
      if (cap_faces < *n_faces) return DCB_ERR_ARG;
      memcpy(faces, r.faces.data(), r.faces.size() * 4);
    }
    return DCB_OK;
  });
}

int dcb_mesh_map(const dcb_batch *b, int buf, int attr_decoder, int which, uint32_t *dst, uint64_t cap, uint64_t *n) {
  return guarded([&]() -> int {
    if (!b || buf < 0 || buf >= (int)b->bufs.size() || !n || which < 0 || which > 3) return DCB_ERR_ARG;
    const BufRec &r = b->bufs[buf];
    if (attr_decoder < 0 || attr_decoder >= (int)r.maps.size() || !r.maps[attr_decoder].set) return DCB_ERR_STATE;
    const MeshMapsHost &m = r.maps[attr_decoder];
    const void *src = which == 0 ? (const void *)m.opposite : which == 1 ? (const void *)m.corner_to_vertex
                    : which == 2 ? (const void *)m.data_to_corner : (const void *)m.vertex_to_data;
    *n = which == 0 ? m.n_corners : which == 1 ? m.n_corners : which == 2 ? m.n_entries : m.n_vertices;
    if (dst) {
      if (cap < *n) return DCB_ERR_ARG;
      memcpy(dst, src, *n * 4);
    }
    return DCB_OK;
  });
}

int dcb_index_finish(dcb_ctx *ctx, dcb_batch *b) {
  return guarded([&]() -> int {
    (void)ctx;
    if (!b) return DCB_ERR_ARG;
    for (Shard &sh : b->shards)
      if (sh.uploaded) return DCB_ERR_STATE;
    // rebuild every shard's stream list with the connectivity-dependent buffers included
    for (Shard &sh : b->shards) {
      sh.streams.clear();
      sh.idx_first = ~0u;
      std::fill(sh.walks.begin(), sh.walks.end(), BufWalk{});
    }
    for (size_t k = 0; k < b->bufs.size(); ++k) {
      BufRec &r = b->bufs[k];
      if (r.pt_failed) {  // the face check runs again for the batch's current order and faces
        r.info.status = DCB_OK;
        r.pt_failed = false;
      }
      if (r.info.needs_connectivity && r.info.status == DCB_OK) {
        if (r.info.attr_section_off == 0) r.info.status = DCB_ERR_CONNECTIVITY;
        r.info.needs_connectivity = 0;
      }
      check_plausible(*b, r);
    parse_attr_section(r, b->shards[r.shard], (int)k, b);
    }
    finalize_layout(b);
    b->conn_done = true;
    return DCB_OK;
  });
}

int dcb_set_output_order(dcb_batch *b, int order) {
  return guarded([&]() -> int {
    if (!b || (order != DCB_ORDER_ENTRIES && order != DCB_ORDER_POINTS)) return DCB_ERR_ARG;
    for (const Shard &sh : b->shards)
      if (sh.uploaded) return DCB_ERR_STATE;
    if (order == b->order) return DCB_OK;
    b->order = order;
    if (b->conn_done) return dcb_index_finish(nullptr, b);
    finalize_layout(b);
    return DCB_OK;
  });
}

int dcb_set_face_output(dcb_batch *b, int mode) {
  return guarded([&]() -> int {
    if (!b || (mode != DCB_FACES_NONE && mode != DCB_FACES_ARENA)) return DCB_ERR_ARG;
    for (const Shard &sh : b->shards)
      if (sh.uploaded) return DCB_ERR_STATE;
    if (mode == b->faces) return DCB_OK;
    // indices dcb_host_connectivity only located for the GPU are not on the host: they need this mode
    for (const BufRec &r : b->bufs)
      if (r.seq_loc.located) return DCB_ERR_STATE;
    b->faces = mode;
    if (b->conn_done) return dcb_index_finish(nullptr, b);
    finalize_layout(b);
    return DCB_OK;
  });
}

int dcb_get_face_info(const dcb_batch *b, int buf, dcb_face_info *out) {
  return guarded([&]() -> int {
    if (!b || !out || buf < 0 || buf >= (int)b->bufs.size()) return DCB_ERR_ARG;
    const BufRec &r = b->bufs[buf];
    memset(out, 0, sizeof *out);
    if (!r.face_src) return DCB_OK;
    out->out_off = b->shards[r.shard].out_base + r.face_off;
    out->out_bytes = 12 * r.n_faces;
    out->n_faces = r.n_faces;
    out->source = r.info.status == DCB_OK ? r.face_src : 0;
    return DCB_OK;
  });
}

int dcb_set_mesh_faces(dcb_batch *b, int buf, const uint32_t *faces, uint64_t n_faces) {
  return guarded([&]() -> int {
    if (!b || buf < 0 || buf >= (int)b->bufs.size()) return DCB_ERR_ARG;
    if ((!faces && n_faces) || n_faces > 0xFFFFFFFFull / 3) return DCB_ERR_ARG;
    BufRec &r = b->bufs[buf];
    if (!r.is_eb) return DCB_ERR_STATE;
    for (const Shard &sh : b->shards)
      if (sh.uploaded) return DCB_ERR_STATE;
    const bool known_before = faces_known(r);
    r.pt_faces = faces;
    r.pt_n_faces = n_faces;
    r.pt_faces_set = true;
    // after dcb_index_finish: re-index only when the buffer's verdict flips (the layout follows the statuses alone)
    if (b->conn_done && b->order == DCB_ORDER_POINTS && !r.info.needs_connectivity && (r.info.status == DCB_OK || r.pt_failed) &&
        point_faces_ok(r, r.info.n_attr_decoders) == r.pt_failed)
      return dcb_index_finish(nullptr, b);
    if (b->conn_done && b->faces == DCB_FACES_ARENA) {  // faces in the arena: a new verdict or a new region size
      if (r.pt_failed || faces_known(r) != known_before) return dcb_index_finish(nullptr, b);
      finalize_layout(b);
    }
    return DCB_OK;
  });
}

int dcb_upload(dcb_ctx *ctx, dcb_batch *b) {
  return guarded([&]() -> int {
    if (!ctx || !b || (int)ctx->devices.size() != b->n_devices) return DCB_ERR_ARG;
    for (const BufRec &r : b->bufs)
      if (r.info.needs_connectivity && r.info.status == DCB_OK) return DCB_ERR_STATE;
    for (int d = 0; d < b->n_devices; ++d) {
      int rc = upload_shard(ctx, b, b->shards[d], d);
      if (!rc) rc = issue_arena_copy(ctx, b, b->shards[d], d);
      if (!rc) rc = issue_maps_copy(ctx, b, b->shards[d], d);
      if (rc) {  // copies and memsets of this and earlier shards may be in flight: nothing may outlive the call
        drain(ctx);
        return rc;
      }
    }
    return sync_all(ctx);
  });
}

int dcb_decode_resident(dcb_ctx *ctx, dcb_batch *b, void *dev_out, void *dev_dbg, uint32_t flags) {
  return guarded([&]() -> int {
    int rc = decode_all(ctx, b, dev_out, dev_dbg, flags);
    if (rc) return rc;
    rc = sync_all(ctx);
    if (rc) return rc;
    absorb_descs(b);
    finish_stats(ctx);
    collect_status(b);
    return DCB_OK;
  });
}

int dcb_download(dcb_ctx *ctx, dcb_batch *b, uint8_t *host_out, uint8_t *host_dbg) {
  return guarded([&]() -> int {
    if (!ctx || !b || (int)ctx->devices.size() != b->n_devices) return DCB_ERR_ARG;
    for (int d = 0; d < b->n_devices; ++d) {
      int rc = download_shard(ctx, b, d, host_out, host_dbg);
      if (rc) return rc;
    }
    return sync_all(ctx);
  });
}

int dcb_decode(dcb_ctx *ctx, dcb_batch *b, uint8_t *host_out, uint8_t *host_dbg, uint32_t flags) {
  return guarded([&]() -> int {
    if (!host_out && b && b->total_out) return DCB_ERR_ARG;
    if ((flags & (DCB_DUMP_SYMBOLS | DCB_DUMP_QINTS)) && !host_dbg) return DCB_ERR_ARG;
    const bool dbg_t = env_flags().debug_timing;
    const auto t0 = std::chrono::steady_clock::now();
    auto ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
    if (!ctx || !b || (int)ctx->devices.size() != b->n_devices) return DCB_ERR_ARG;
    int rc = decode_all(ctx, b, nullptr, nullptr, flags, host_out, host_dbg);
    if (rc) return rc;
    const double t_dec = ms();
    rc = sync_all(ctx);
    if (rc) return rc;
    if (dbg_t) fprintf(stderr, "[dcb timing] decode_all issued %.1f ms, download done %.1f ms\n", t_dec, ms());
    absorb_descs(b);
    finish_stats(ctx);
    collect_status(b);
    return DCB_OK;
  });
}

int dcb_decode_scatter(dcb_ctx *ctx, dcb_batch *b, uint8_t *const *outs, int n_outs, uint32_t flags) {
  return guarded([&]() -> int {
    if (!outs && n_outs) return DCB_ERR_ARG;
    if (b && b->faces == DCB_FACES_ARENA) return DCB_ERR_STATE;  // no slot for the faces
    int rc = decode_all(ctx, b, nullptr, nullptr, flags & ~(DCB_DUMP_SYMBOLS | DCB_DUMP_QINTS));
    if (rc) return rc;
    int k = 0;
    for (const BufRec &r : b->bufs) {
      const Shard &sh = b->shards[r.shard];
      const BufWalk &w = sh.walks[r.local];
      CUDA_TRY(cudaSetDevice(sh.device));
      for (int i = 0; i < w.stream_count; ++i, ++k) {
        if (k >= n_outs) break;
        const size_t si = (size_t)w.stream_first + i;
        if (outs[k] && sh.fin_bytes[si] && r.info.status == DCB_OK && w.status == DCB_OK)
          CUDA_TRY(cudaMemcpyAsync(outs[k], sh.ext_out + sh.fin_off[si], sh.fin_bytes[si], cudaMemcpyDeviceToHost,
                                   ctx->streams[r.shard]));
      }
    }
    rc = sync_all(ctx);
    if (rc) return rc;
    absorb_descs(b);
    finish_stats(ctx);
    collect_status(b);
    return DCB_OK;
  });
}

void *dcb_device_out(const dcb_batch *b, int dev_index) {
  if (!b || dev_index < 0 || dev_index >= (int)b->shards.size()) return nullptr;
  return b->shards[dev_index].ext_out;
}

int dcb_sync(dcb_ctx *ctx) { return ctx ? sync_all(ctx) : DCB_ERR_ARG; }

int dcb_status(const dcb_batch *b, int buf) {
  if (!b || buf < 0 || buf >= (int)b->bufs.size()) return DCB_ERR_ARG;
  return b->bufs[buf].info.status;
}

void dcb_batch_free(dcb_batch *b) {
  if (!b) return;
  for (Shard &sh : b->shards) free_shard_device(sh);
  delete b;
}

int dcb_last_stats(const dcb_ctx *ctx, dcb_launch_stats *out) {
  if (!ctx || !out) return DCB_ERR_ARG;
  *out = ctx->stats;
  return DCB_OK;
}

}  // extern "C"
