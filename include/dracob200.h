/*
 * include/dracob200.h -- C ABI of libdracob200.so: batch Draco attribute decode on B200 (sm_100a).
 *
 * This is the drop-in boundary for the attribute-decode hot path of B3zaleel/draco-sharp.  The
 * reference has no FFI seam: `DracoDecoder` is a concrete class (src/Draco/IO/DracoDecoder.cs:8,14,19)
 * that decodes one buffer on one CPU thread.  A C# `DracoBatchDecoder` (csharp/DracoBatchDecoder.cs,
 * shown in INTEGRATION.md) P/Invokes exactly the entry points below; Python (ctypes) and C++ callers
 * use the same calls.  All structs are POD, little-endian, pointer-free inside arrays (blittable).
 *
 * What each entry point replaces in the reference (per buffer, per attribute):
 *   dcb_index        DracoDecoder.DecodeHeader (DracoDecoder.cs:44-64), ConnectivityDecoder.DecodeAttributes
 *                    phases 1-3 (ConnectivityDecoder.cs:16-39), AttributesDecoder.DecodeAttributesData
 *                    (Attributes/AttributesDecoder.cs:19-63), SequentialAttributeDecodersController
 *                    .DecodeAttributesData (:16-27) and the field reads of SequentialIntegerAttributeDecoder
 *                    .DecodeValues (Attributes/SequentialIntegerAttributeDecoder.cs:23-44,61) -- header
 *                    bytes only, never symbol payloads.
 *   dcb_set_mesh_maps  the inputs of MeshPredictionSchemeData (Attributes/PredictionSchemes/
 *                    MeshPredictionSchemeData.cs:5-24): CornerTable.{Opposite,Vertex} (Mesh/CornerTable.cs:9-12)
 *                    and MeshAttributeIndicesEncodingData (Attributes/MeshAttributeIndicesEncodingData.cs:5-19),
 *                    produced on the host by Edgebreaker connectivity decoding.
 *   dcb_decode*      the hot path itself, on the GPU: SymbolDecoding.DecodeSymbols (Entropy/SymbolDecoding.cs:7-67),
 *                    RAnsSymbolDecoder.Create/StartDecoding (Entropy/RAnsSymbolDecoder.cs:12-59), RAnsDecoder
 *                    .ReadInit/Read/BuildLookupTable (Entropy/RAnsDecoder.cs:20-99), BitUtilities
 *                    .ConvertSymbolsToSignedInts (BitUtilities.cs:94-103), PredictionSchemeDeltaDecoder
 *                    .ComputeOriginalValues (…/PredictionSchemeDeltaDecoder.cs:23-37), MeshPredictionScheme
 *                    ParallelogramDecoder.ComputeOriginalValues (…:29-89), the wrap and octahedron decoding
 *                    transforms, AttributeQuantizationTransform.InverseTransformAttribute
 *                    (Attributes/AttributeQuantizationTransform.cs:179-199), AttributeOctahedronTransform
 *                    .InverseTransformAttribute (Attributes/AttributeOctahedronTransform.cs:82-102) and
 *                    SequentialIntegerAttributeDecoder.StoreTypedValues (…:142-160).
 *   dcb_status       the reference's exceptions (Extensions/Assertions.cs:5-24 -> InvalidDataException,
 *                    EndOfStreamException, NotImplementedException), as per-buffer integer codes: one
 *                    malformed buffer never poisons the batch and no C++ exception crosses the ABI.
 *
 * There is NO CPU fallback: every dcb_decode* call fails with DCB_ERR_NO_DEVICE when no sm_100 GPU is
 * usable.  Ownership: the caller owns input and output memory; the library owns ctx and batch objects.
 * Threading: calls on one ctx are serialised by the caller; distinct ctxs may run concurrently.
 */
#ifndef DRACOB200_H
#define DRACOB200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define DCB_VERSION 100 /* 0.1.0 */

/* per-buffer / per-call status codes (mirror the reference's exception sites) */
enum {
  DCB_OK = 0,
  DCB_ERR_EOF = -1,          /* EndOfStreamException (BinaryReader) */
  DCB_ERR_MAGIC = -2,        /* DracoDecoder.cs:47-50 */
  DCB_ERR_UNSUPPORTED = -3,  /* NotImplemented/NotSupported: kd-tree point clouds, version != 2.2, out-of-scope predictors */
  DCB_ERR_SCHEME = -4,       /* SymbolDecoding.cs:26 */
  DCB_ERR_BITLEN = -5,       /* SymbolDecoding.cs:56 */
  DCB_ERR_TABLE = -6,        /* RAnsSymbolDecoder.cs:31, RAnsDecoder.cs:80,87 */
  DCB_ERR_RANS_INIT = -7,    /* RAnsDecoder.cs:22,33,39,53 */
  DCB_ERR_PRED = -8,         /* SequentialIntegerAttributeDecoder.cs:26,31 */
  DCB_ERR_WRAP = -9,         /* PredictionSchemeWrapDecodingTransform.cs:73, PredictionSchemeWrapTransform.cs:91 */
  DCB_ERR_QUANT = -10,       /* AttributeQuantizationTransform.cs:121, OctahedronToolBox.cs:15 */
  DCB_ERR_ATTR = -11,        /* AttributesDecoder.cs:37-39, SequentialNormalAttributeDecoder.cs:14-15 */
  DCB_ERR_TAG = -12,         /* DecoderBuffer.cs:141 */
  DCB_ERR_NUM_SYMBOLS = -13, /* SymbolDecoding.cs:36,59 */
  DCB_ERR_MAPS = -14,        /* mesh prediction without / with inconsistent connectivity maps */
  DCB_ERR_CONNECTIVITY = -15,
  /* call-level errors (never stored as a buffer status) */
  DCB_ERR_ARG = -100,
  DCB_ERR_NO_DEVICE = -101,  /* no usable sm_100 device: there is no CPU fallback */
  DCB_ERR_CUDA = -102,
  DCB_ERR_OOM = -103,
  DCB_ERR_STATE = -104       /* call order violated (e.g. decode before upload, mesh maps missing) */
};

typedef struct dcb_ctx dcb_ctx;     /* one per process or per GPU set */
typedef struct dcb_batch dcb_batch; /* one per indexed batch of buffers */

typedef struct dcb_buffer_info {
  int32_t status;          /* DCB_OK or the first error met while indexing */
  int32_t geometry_type;   /* 0 point cloud, 1 triangular mesh (DracoHeader.EncoderType) */
  int32_t encoder_method;  /* 0 sequential, 1 Edgebreaker */
  int32_t version_major, version_minor;
  int32_t flags;
  uint32_t n_points;       /* point clouds / sequential meshes; 0 until known for Edgebreaker */
  int32_t n_attr_decoders;
  int32_t n_attrs;
  int32_t needs_connectivity; /* 1: host must call dcb_set_mesh_maps before decode */
  int32_t device;          /* device index (into the ctx's list) this buffer was sharded to */
  int32_t reserved;
  uint64_t attr_section_off;  /* byte offset of the ATTRIBUTES section (mesh: set by dcb_set_attr_section) */
} dcb_buffer_info;

typedef struct dcb_attr_info {
  int32_t att_type;       /* GeometryAttributeType: 0 position 1 normal 2 color 3 texcoord 4 generic */
  int32_t data_type;      /* DataType enum value (UInt8 = 2 ... Float32 = 9) */
  int32_t num_components;
  int32_t normalized;
  uint32_t unique_id;
  int32_t seq_decoder_type; /* 0 generic 1 integer 2 quantization 3 normals */
  int32_t decoder_id;
  int32_t pred_method;    /* PredictionSchemeMethod, -2 none; decoded on the GPU: 0 difference, 1 parallelogram, 4 constrained
                             multi-parallelogram, 5 tex-coords-portable, 6 geometric normal (2, 3: pre-2.2 streams, UNSUPPORTED) */
  int32_t transform;      /* PredictionSchemeTransformType, -1 none */
  int32_t scheme;         /* 0 tagged 1 raw -1 n/a */
  int32_t precision_bits;
  uint32_t n_entries;     /* UniqueEntriesCount */
  uint64_t out_bytes;     /* rows * num_components * sizeof(data_type); rows = n_entries, or n_points for Edgebreaker
                             meshes in DCB_ORDER_POINTS */
  uint64_t out_off;       /* offset of this attribute inside the batch output arena (128-byte aligned) */
  uint64_t dbg_off;       /* offset inside the debug arena (int32 per portable value), if requested */
  int32_t xf_a, xf_b;     /* wrap min/max or oct max_quantized_value/center_value */
  float q_min[4];
  float q_range;
  int32_t q_bits;
  int32_t resolved;       /* 0 while the attribute lies behind an undecoded Tagged bit area */
} dcb_attr_info;

/* decode flags */
#define DCB_DUMP_SYMBOLS 1u /* debug arena receives the decoded symbols (uint32) */
#define DCB_DUMP_QINTS 2u   /* debug arena receives the portable integers after prediction (int32) */

int dcb_version(void);
int dcb_device_count(void);
const char *dcb_error_string(int code);

/* device_ids == NULL / n_devices == 0: use the current CUDA device only.
 * Distinct ids: a batch is sharded by buffer across the GPUs (longest-processing-time-first on compressed bytes; no
 * collective, SURVEY 8e).  The SAME id listed K times: K pipeline slices on that GPU -- contiguous runs of buffers with
 * their own streams and arenas, so that in a host-buffer decode (dcb_decode / dcb_decode_scatter) slice k decodes while
 * slice k+1 uploads and slice k-1 downloads.  The context caches the device arenas of freed batches. */
int dcb_create(const int *device_ids, int n_devices, dcb_ctx **out);
void dcb_destroy(dcb_ctx *ctx);
/* Launch on a caller-owned CUDA stream (cudaStream_t) of device `dev_index` instead of the ctx's own. */
int dcb_set_stream(dcb_ctx *ctx, int dev_index, void *cuda_stream);

/* Plausibility limits of ONE buffer, applied while indexing (before any arena is sized): a buffer whose header
 * claims more points (or, for meshes, more attribute entries) than
 *     max_points_per_buffer            (0 = no absolute cap), or
 *     65536 + points_per_byte * length (0 = unchecked; default 4096)
 * gets DCB_ERR_ATTR on its own and reserves nothing, instead of inflating the whole batch.  The reference has no
 * such check -- it allocates what the header says (PointCloud.cs, DataBuffer.cs) and dies of it. */
int dcb_set_limits(dcb_ctx *ctx, uint64_t max_points_per_buffer, uint64_t points_per_byte);

/* Phase 1 (host, O(header bytes)): parse containers, locate every stream.  Never reads payloads.
 * The buffers must stay valid until dcb_upload/dcb_decode has returned. */
int dcb_index(dcb_ctx *ctx, const uint8_t *const *bufs, const uint64_t *lens, int n_bufs, dcb_batch **out);
/* Same, for buffers packed in one arena (one host->device copy instead of n). */
int dcb_index_arena(dcb_ctx *ctx, const uint8_t *arena, const uint64_t *offs, const uint64_t *lens, int n_bufs,
                    dcb_batch **out);
int dcb_get_buffer_info(const dcb_batch *b, int buf, dcb_buffer_info *out);
int dcb_get_attr_info(const dcb_batch *b, int buf, int attr, dcb_attr_info *out);
uint64_t dcb_batch_out_bytes(const dcb_batch *b);  /* size of the output arena, all devices */
uint64_t dcb_batch_dbg_bytes(const dcb_batch *b);  /* size of the debug arena */
uint64_t dcb_batch_in_bytes(const dcb_batch *b);   /* compressed bytes that travel host->device */
uint64_t dcb_batch_points(const dcb_batch *b);     /* sum of n_points over OK buffers */
/* algorithmic bytes of the decode (payload + table + bit area + header + map reads + outputs; SURVEY 8d) */
uint64_t dcb_batch_algo_bytes(const dcb_batch *b);

/* Mesh only: where ATTRIBUTES starts (the host decoded connectivity up to there) and, per attributes
 * decoder, the entry count + connectivity-derived arrays.  The four arrays are BORROWED, not copied: they
 * must stay valid and unchanged until the dcb_decode* / dcb_upload call that consumes them has returned
 * (56 bytes per vertex that the library reads exactly once, for the host->device copy; page-locked arrays
 * travel at full PCIe speed, pageable ones through the driver's staging).  n_corners must be a multiple of 3. */
int dcb_set_attr_section(dcb_batch *b, int buf, uint64_t attr_section_off, uint32_t n_points);
int dcb_set_mesh_maps(dcb_batch *b, int buf, int attr_decoder, const uint32_t *opposite,
                      const uint32_t *corner_to_vertex, uint64_t n_corners, const uint32_t *data_to_corner,
                      uint64_t n_entries, const int32_t *vertex_to_data, uint64_t n_vertices);
/* Host helper for callers without the C# host (SURVEY 8f-1): decodes the Edgebreaker connectivity of mesh buffer
 * `buf` ON THE CPU -- the part of the reference that stays on the host, MeshEdgeBreakerDecoder.DecodeConnectivity
 * (Mesh/MeshEdgeBreakerDecoder.cs:25-638), the standard / valence traversal decoders and the depth-first attribute
 * traversal (Mesh/Traverser/DepthFirstTraverser.cs:9-99) -- and installs what dcb_set_attr_section +
 * dcb_set_mesh_maps would.  A buffer whose connectivity is invalid or unsupported gets its own status. */
int dcb_host_connectivity(dcb_batch *b, int buf);
/* Faces (3 point ids each) of a mesh decoded by dcb_host_connectivity (Mesh.SetFace, MeshEdgeBreakerDecoder.cs:622-636).
 * faces == NULL: only *n_faces is written.  DCB_ERR_STATE for a sequential mesh whose indices the GPU decodes into the
 * output arena (DCB_FACES_ARENA): they are not on the host. */
int dcb_mesh_faces(const dcb_batch *b, int buf, uint32_t *faces, uint64_t cap_faces, uint64_t *n_faces);
/* Read back one installed map of an attributes decoder: which = 0 opposite, 1 corner_to_vertex, 2 data_to_corner,
 * 3 vertex_to_data (int32 bit patterns).  dst == NULL: only *n is written.  What a host needs to build the
 * reference's CornerTable / MeshAttributeIndicesEncodingData from dcb_host_connectivity's result. */
int dcb_mesh_map(const dcb_batch *b, int buf, int attr_decoder, int which, uint32_t *dst, uint64_t cap, uint64_t *n);
/* Re-run the attribute indexing of mesh buffers once their maps are set. */
int dcb_index_finish(dcb_ctx *ctx, dcb_batch *b);

/* Output order of a batch.
 *   DCB_ORDER_ENTRIES (default): every attribute holds its unique values in entry order -- the order the encoder's
 *       traversal visited them (n_entries rows, PointAttribute with a point-to-value map in the reference).
 *   DCB_ORDER_POINTS: every attribute of an Edgebreaker mesh holds n_points rows, row p being the value of the entry
 *       the reference maps point p to (MeshTraversalSequencer.UpdatePointToAttributeIndexMapping,
 *       MeshTraversalSequencer.cs:33-51): for each attributes decoder d, for each corner c in increasing order,
 *           p = faces[c]; v = corner_to_vertex_d[c]; e = vertex_to_data_d[v]; map_d[p] = e
 *       The last corner of a point wins.  p >= n_points, v >= the decoder's vertex count or e outside [0, n_entries)
 *       fail that buffer alone with DCB_ERR_MAPS; a point no corner references gets zero bytes.  Each attribute uses
 *       the maps of its own decoder.  The gather runs on the GPU.  Point clouds and sequential meshes map points to
 *       entries one to one: their bytes are the same in both orders.  The debug arena (DCB_DUMP_*) stays in entry order.
 * dcb_attr_info.out_off / out_bytes describe what lands in the output arena, so rows = out_bytes / (num_components *
 * sizeof(type)); n_entries keeps its meaning.  dcb_batch_out_bytes is the size of the arena in the chosen order. */
#define DCB_ORDER_ENTRIES 0
#define DCB_ORDER_POINTS 1
/* Before the first dcb_upload / dcb_decode* of the batch (DCB_ERR_STATE afterwards); re-lays out the output arena. */
int dcb_set_output_order(dcb_batch *b, int order);
/* Edgebreaker meshes whose connectivity the caller decoded: Mesh.Faces as 3 point ids per face, BORROWED like the
 * maps (valid until the decode / upload that consumes them returns).  faces == NULL && n_faces == 0: the mesh has no
 * attribute seams, point ids are vertex ids, faces = corner_to_vertex of attributes decoder 0 (AssignPointsToCorners
 * without attribute data) -- nothing extra travels to the device.  dcb_host_connectivity installs its own faces.
 * In point order an Edgebreaker buffer without faces, or whose 3 * n_faces is not the corner count of each of its
 * decoders, fails with DCB_ERR_MAPS.  Point clouds and sequential meshes: DCB_ERR_STATE.  Install faces before
 * dcb_index_finish, like the maps: afterwards, a call that turns a buffer's verdict (DCB_ERR_MAPS <-> ok) re-runs the
 * attribute indexing of the whole batch. */
int dcb_set_mesh_faces(dcb_batch *b, int buf, const uint32_t *faces, uint64_t n_faces);

/* Faces of meshes in the output arena.
 *   DCB_FACES_NONE (default): faces stay on the host (dcb_mesh_faces); the arena holds attributes only.
 *   DCB_FACES_ARENA: every mesh buffer that is ok after dcb_index_finish gets a faces region in the output arena:
 *       3 u32 point ids per face (Mesh.Faces, the ids dcb_mesh_faces returns), behind the attributes of its shard, on a
 *       128-byte boundary.  dcb_batch_out_bytes includes the regions; attribute out_off / out_bytes keep their meaning.
 *       Independent of the output order: in DCB_ORDER_POINTS, values[faces] is the triangle soup, on the device.
 *   Where the faces come from:
 *     Edgebreaker    the faces installed by dcb_host_connectivity or dcb_set_mesh_faces (the NULL form: corner_to_vertex
 *                    of attributes decoder 0); they travel with the maps and are copied into the region on the device.
 *                    A buffer without faces fails with DCB_ERR_MAPS at dcb_index_finish.
 *     sequential     dcb_host_connectivity called while the batch is in this mode.  Plain indices (connectivity
 *                    method 1: 1, 2 or 4 bytes, or varints for 65536 <= points < 2^21) are only LOCATED on the host --
 *                    framing errors give the statuses the host decode gives -- and decoded on the GPU; so are Raw index
 *                    differences (method 0): one more Raw rANS stream, then a scan that fails the buffer alone with
 *                    DCB_ERR_CONNECTIVITY when an index drops below 0 or passes INT32_MAX.  dcb_mesh_faces then returns
 *                    DCB_ERR_STATE.  Tagged index differences cannot be located without decoding them (their bit area
 *                    has no length prefix, SymbolDecoding.cs:37-49): they are decoded on the host as before and travel
 *                    with the maps.  A sequential buffer whose connectivity the caller installed with
 *                    dcb_set_attr_section has no faces: DCB_ERR_MAPS.
 *   dcb_decode_scatter has no slot for faces: DCB_ERR_STATE for a batch in this mode. */
#define DCB_FACES_NONE 0
#define DCB_FACES_ARENA 1
/* Before the first dcb_upload / dcb_decode* of the batch (DCB_ERR_STATE afterwards); re-lays out the output arena.
 * Set it before dcb_host_connectivity for the sequential indices to be decoded on the GPU; once dcb_host_connectivity has
 * located indices for the GPU, turning the mode off fails with DCB_ERR_STATE (those faces are not on the host). */
int dcb_set_face_output(dcb_batch *b, int mode);
typedef struct dcb_face_info {
  uint64_t out_off;    /* offset of the faces region in the output arena, 128-byte aligned */
  uint64_t out_bytes;  /* 12 * n_faces: u32 point ids, 3 per face */
  uint64_t n_faces;
  int32_t source;      /* 0 none (point cloud, failed buffer, mode off), 1 decoded on the host, 2 decoded on the GPU */
  int32_t reserved;
} dcb_face_info;
/* All zero for a batch in DCB_FACES_NONE and for buffers without a faces region. */
int dcb_get_face_info(const dcb_batch *b, int buf, dcb_face_info *out);

/* Phase 2 (device).  One-call form: host->device copy, kernels, device->host copy.
 * host_out: one arena of dcb_batch_out_bytes() bytes laid out by dcb_attr_info.out_off; host_dbg may be
 * NULL unless a DUMP flag is set. */
int dcb_decode(dcb_ctx *ctx, dcb_batch *b, uint8_t *host_out, uint8_t *host_dbg, uint32_t flags);
/* Same, writing each attribute to its own caller pointer (outs[k] for the k-th attribute in
 * (buffer, attribute) order over all buffers; NULL entries are skipped). */
int dcb_decode_scatter(dcb_ctx *ctx, dcb_batch *b, uint8_t *const *outs, int n_outs, uint32_t flags);

/* Split form, for callers that keep data on the device:
 *   upload   : compressed bytes + descriptors -> HBM
 *   resident : kernels only; outputs stay in HBM.  dev_out/dev_dbg: device pointers for single-device ctxs
 *              (NULL = library-owned arenas, see dcb_device_out)
 *   download : device -> host of the output arena */
int dcb_upload(dcb_ctx *ctx, dcb_batch *b);
int dcb_decode_resident(dcb_ctx *ctx, dcb_batch *b, void *dev_out, void *dev_dbg, uint32_t flags);
int dcb_download(dcb_ctx *ctx, dcb_batch *b, uint8_t *host_out, uint8_t *host_dbg);
void *dcb_device_out(const dcb_batch *b, int dev_index);
int dcb_sync(dcb_ctx *ctx);

int dcb_status(const dcb_batch *b, int buf); /* 0 ok; <0 error code */
void dcb_batch_free(dcb_batch *b);

/* Introspection for benchmarks: kernels launched by the last dcb_decode* call and their device time. */
typedef struct dcb_launch_stats {
  int32_t n_launches;        /* kernels launched by the last decode */
  int32_t n_streams;         /* rANS streams decoded */
  int32_t n_waves;           /* residency waves of the dominant rANS kernel */
  int32_t lanes_per_warp;
  uint64_t smem_per_stream;  /* bytes of shared memory per resident stream (dominant kernel) */
  float ms_total;            /* CUDA-event time of all kernels of the last decode (device 0) */
  float ms_dominant;         /* CUDA-event time of the dominant kernel (largest share of ms_total) */
  float ms_raw;              /* largest Raw rANS fused kernel */
  float ms_tag;              /* tag rANS kernels + walk resolve (Tagged streams) */
  float ms_par;              /* point-parallel bit extraction / scan / store passes (Tagged, uncompressed) */
  float ms_para;             /* parallelogram dependency + chain kernels (mesh attributes) */
  uint64_t algo_bytes_dominant; /* algorithmic bytes of the dominant kernel (compulsory reads + writes) */
  char dominant_name[96];
} dcb_launch_stats;
int dcb_last_stats(const dcb_ctx *ctx, dcb_launch_stats *out);

#ifdef __cplusplus
}
#endif
#endif
