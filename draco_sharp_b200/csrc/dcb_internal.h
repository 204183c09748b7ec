// draco_sharp_b200/csrc/dcb_internal.h -- structures shared by the host indexer, the C-ABI layer
// and the sm_100a kernels of libdracob200.so.  Product code: nothing here touches oracle/.
#pragma once
#include <stdint.h>

#include "../../include/dracob200.h"

#if defined(__CUDACC__)
#define DCB_HD __host__ __device__ __forceinline__
#else
#define DCB_HD inline
#endif

// DCB_FACES_ARENA: bytes of a varint index run per checkpoint = one CTA iteration of seq_varint_kernel (dcb_faces.cu)
#define DCB_VARINT_CHUNK 4096u

// wire enums (numeric values are part of the bitstream; src/Draco/IO/Enums/*.cs)
enum : int32_t {
  DT_INT8 = 1, DT_UINT8 = 2, DT_INT16 = 3, DT_UINT16 = 4, DT_INT32 = 5, DT_UINT32 = 6,
  DT_INT64 = 7, DT_UINT64 = 8, DT_FLOAT32 = 9, DT_FLOAT64 = 10, DT_BOOL = 11, DT_COUNT = 12
};
enum : int32_t { SEQ_GENERIC = 0, SEQ_INTEGER = 1, SEQ_QUANTIZATION = 2, SEQ_NORMALS = 3 };
enum : int32_t {
  PRED_NONE = -2, PRED_DIFFERENCE = 0, PRED_PARALLELOGRAM = 1, PRED_CONSTRAINED_MULTI = 4, PRED_TEX_COORDS_PORTABLE = 5,
  PRED_GEOMETRIC_NORMAL = 6, PRED_COUNT = 7
};
enum : int32_t { XF_NONE = -1, XF_DELTA = 0, XF_WRAP = 1, XF_OCT = 2, XF_OCT_CANON = 3, XF_COUNT = 4 };
// symbol source of a stream
enum : uint8_t {
  SCHEME_TAGGED = 0,      // SymbolDecoding.cs:30-50
  SCHEME_RAW = 1,         // SymbolDecoding.cs:52-67
  SCHEME_EMPTY = 253,     // zero values: nothing is read (SymbolDecoding.cs:9-13)
  SCHEME_GENERIC = 254,   // PORTABLE(generic): n x byte_stride raw bytes (SequentialAttributeDecoder.cs:75-86)
  SCHEME_UNCOMPRESSED = 255  // compressed == 0: num_bytes per value (SequentialIntegerAttributeDecoder.cs:68-84)
};

// how the portable integers of a stream are reconstructed from corrections
enum : uint8_t {
  RECON_NONE = 0,          // no prediction scheme object: values = zig-zag(symbols)
  RECON_DELTA_WRAP = 1,    // PredictionSchemeDeltaDecoder + wrap transform
  RECON_DELTA_OCT = 2,     // PredictionSchemeDeltaDecoder + octahedron transform (non canonical)
  RECON_DELTA_OCT_CANON = 3,
  RECON_PARA_WRAP = 4      // a mesh prediction scheme + wrap transform: the symbol kernels leave the corrections in the stream's
                           // scratch and a chain kernel follows -- MeshPredictionSchemeParallelogramDecoder (pred_method
                           // PRED_PARALLELOGRAM), MeshPredictionSchemeConstrainedMultiParallelogramDecoder (PRED_CONSTRAINED_MULTI)
                           // or MeshPredictionSchemeTexCoordsPortableDecoder (PRED_TEX_COORDS_PORTABLE)
  ,
  RECON_GEO_OCT = 5,       // MeshPredictionSchemeGeometricNormalDecoder + octahedron transform: the symbol kernels leave the
  RECON_GEO_OCT_CANON = 6  // corrections in the stream's scratch, geo_normal_kernel (point-parallel) finishes the attribute
};
// how portable integers become attribute bytes
enum : uint8_t {
  STORE_DEQUANT = 0,  // AttributeQuantizationTransform.InverseTransformAttribute -> float32 x nc
  STORE_OCT_UNIT = 1, // AttributeOctahedronTransform.InverseTransformAttribute  -> float32 x 3
  STORE_NARROW = 2,   // StoreTypedValues<T>: low sizeof(T) bytes of each int32
  STORE_COPY = 3      // generic attribute: raw bytes
};
// walk progress of one attribute
enum : uint8_t {
  ST_UNPARSED = 0,
  ST_TAGS_PENDING = 1,  // Tagged: table + payload located, bit area length unknown until the tags are decoded
  ST_PORTABLE = 2,      // PORTABLE fully located (incl. PRED_DATA)
  ST_READY = 3          // XFORM_PARAMS read too: the stream can be decoded end to end
};

// One attribute of one buffer.  Offsets are absolute byte offsets into the device input arena of
// the shard that owns the buffer.
struct StreamDesc {
  uint64_t buf_begin, buf_end;   // the owning .drc buffer inside the arena
  uint64_t table_off;            // first byte of RANS_TABLE (the num_symbols varint)
  uint64_t payload_off;          // first byte of the rANS payload
  uint64_t payload_len;
  uint64_t bits_off;             // Tagged: first byte of the LSB-first bit area
  uint64_t raw_off;              // uncompressed ints / generic: first value byte
  uint64_t out_off;              // output arena offset of the attribute
  uint64_t out_bytes;
  uint64_t dbg_off;              // debug arena offset (int32 per portable value)
  uint64_t aux_off;              // scratch arena offset (corrections int32[nv]), 16-byte aligned
  uint64_t tag_off;              // scratch arena offset (tags u8[n] then u32 chunk sums), 16-byte aligned
  uint64_t map_off[4];           // parallelogram: opposite, corner_to_vertex, data_to_corner, vertex_to_data
  uint64_t bits_total;           // device-written: bits consumed in the Tagged bit area
  uint64_t orient_off;           // tex coords: first byte (prob_zero) of the rABS-coded orientation flags; geometric normal: of the flip bits
  uint64_t crease_off[4];        // constrained multi-parallelogram: first byte (prob_zero) of the rABS-coded crease flags of
                                 // context c (entries with c + 1 parallelograms); meaningless when n_crease[c] == 0
  uint32_t n_crease[4];          // ... and their number
  uint32_t n_orient;             // tex coords: number of orientation flags; geometric normal: number of flip bits (= entries)
  int32_t parent;                // tex coords: shard-wide stream index of the buffer's position attribute, or -1
  uint32_t n_corners, n_vertices;
  uint32_t n_entries;
  uint32_t num_symbols;          // table alphabet size
  uint32_t n_active;             // symbols with non-zero probability
  uint32_t dense_prefix;         // leading symbols 0..dense_prefix-1 all have non-zero probability
  uint32_t unique_id;
  int32_t xf_a, xf_b;            // wrap min,max | oct max_quantized_value, center
  float q_min[4];
  float q_range;
  int32_t q_bits;
  int32_t buf_index, attr_index; // position in the batch (attr_index is relative to the buffer)
  int32_t status;                // device-written DCB_ERR_* (0 = ok)
  int32_t irregular;             // device-written: delta+wrap stream that needs the serial recurrence
  int8_t pred_method, transform;
  uint8_t nc, ncp;               // attribute components / portable components
  uint8_t scheme;                // SCHEME_*
  uint8_t prec_bits, max_bit_length;
  uint8_t recon, store;
  uint8_t data_type;             // output DataType
  uint8_t att_type, normalized, seq_type, decoder_id;
  uint8_t zigzag;
  uint8_t raw_num_bytes;         // uncompressed: bytes per value
  uint8_t state;                 // ST_*
  uint8_t compressed;
  uint8_t has_maps;              // host supplied connectivity maps for this attribute's decoder
  uint8_t pad_[1];
  // narrow_blk[k] (k = 1..7): 128-slot block holding the first table entry narrower than 2^k slots (2^prec >> 7 when
  // there is none) -- what the launch planner needs to size the narrow region of the two-region LUT
  uint16_t narrow_blk[8];
  // bucket-record kernels (dcb_rans_rec.cu): 8-byte units of table memory a lane needs, per candidate bucket size of the
  // wide region (2^(DCB_REC_KA0 + j) slots); 0xFFFF = the table does not have the shape (see walk_rans_table)
  uint16_t rec_need[4];
};

// Resumable container walk of one buffer (runs on the host; continues on the device behind Tagged
// bit areas, whose length is only known once the tags are decoded).
struct BufWalk {
  uint64_t begin, end;      // arena offsets of this buffer
  uint64_t pos;             // where the walk continues
  int32_t status;
  int32_t stream_first, stream_count;
  int32_t cur;              // relative index of the stream being parsed
  int32_t dec_start;        // relative index of the first stream of the current attributes decoder
  int32_t phase;            // 0 PORTABLE pass, 1 XFORM_PARAMS pass, 2 done
  int32_t blocked;          // relative stream index whose Tagged bit area blocks the walk, or -1
  uint8_t geom_type, method, pad_[2];
};

DCB_HD int dcb_dtype_len(int dt) {
  switch (dt) {
    case DT_INT8: case DT_UINT8: case DT_BOOL: return 1;
    case DT_INT16: case DT_UINT16: return 2;
    case DT_INT32: case DT_UINT32: case DT_FLOAT32: return 4;
    case DT_INT64: case DT_UINT64: case DT_FLOAT64: return 8;
    default: return -1;
  }
}
// RAnsSymbolCoding.cs:10-26
DCB_HD int dcb_rans_precision(int max_bit_length) {
  int p = 3 * max_bit_length / 2;
  return p < 12 ? 12 : (p > 20 ? 20 : p);
}

// ---- bucket-record tables (dcb_rans_rec.cu) ----
// The slot axis [0, 2^prec) of a table is cut at ta <= tb <= tc:
//   [0, ta)        one 8-byte record per 2^ka slots     every such bucket meets at most two table entries below ta
//   [ta, tb)       one record per 16 slots              likewise below tb
//   [tb, tc)       one record per 8 slots               likewise below tc
//   [tc, 2^prec)   one byte per slot                    every entry reaching into it is at most 16 slots wide, and
//                                                       starts at or behind tc
// then a bitmap of entry starts over the byte region (u32 words) with a u16 running count per word.  The value map of
// the table follows (planned separately).  A bucket meets at most two entries iff at most one entry boundary lies
// strictly inside it; RecShape finds, while the table streams by, for every bucket size the second boundary of the
// first bucket that breaks the rule (records of that size are good for all slots in front of it) and the end of the
// last entry wider than 16 slots, and from them the cuts.  Host (container walk -> launch planner) and device (table
// build) run the same code on the same bytes.
#define DCB_REC_KA0 5
struct RecLayout {
  uint32_t n_a, n_b, n_b2, n_c;                     // records / records / records / bytes
  uint32_t off_b, off_b2, off_c, off_bm, off_cnt;   // byte offsets inside the lane's area (records first: 8-byte aligned)
  uint32_t bytes;                                   // multiple of 8
};
DCB_HD RecLayout dcb_rec_layout(uint32_t ta, uint32_t tb, uint32_t tc, uint32_t prec, uint32_t ka) {
  RecLayout l;
  l.n_a = (ta + (1u << ka) - 1u) >> ka;
  l.n_b = tb > ta ? ((tb + 15u) >> 4) - (ta >> 4) : 0u;
  l.n_b2 = tc > tb ? ((tc + 7u) >> 3) - (tb >> 3) : 0u;
  l.n_c = prec - tc;
  l.off_b = 8u * l.n_a;
  l.off_b2 = l.off_b + 8u * l.n_b;
  l.off_c = l.off_b2 + 8u * l.n_b2;
  l.off_bm = (l.off_c + l.n_c + 3u) & ~3u;
  const uint32_t words = (l.n_c + 31u) >> 5;
  l.off_cnt = l.off_bm + 4u * words;
  l.bytes = (l.off_cnt + 2u * words + 7u) & ~7u;
  return l;
}
struct RecShape {
  // bucket sizes 2^3, 2^4, 2^DCB_REC_KA0 .. 2^(DCB_REC_KA0 + 3)
  uint32_t bad_at[6];      // second boundary inside the first bucket holding two (0xFFFFFFFF: none)
  uint32_t prev_bucket[6]; // bucket of the last boundary seen that lies strictly inside one
  uint32_t end_wide;       // end of the last entry wider than 16 slots
  DCB_HD static uint32_t scale(int j) { return j < 2 ? 3u + (uint32_t)j : (uint32_t)(DCB_REC_KA0 + j - 2); }
  DCB_HD void begin() {
    for (int j = 0; j < 6; ++j) {
      bad_at[j] = 0xFFFFFFFFu;
      prev_bucket[j] = 0xFFFFFFFFu;
    }
    end_wide = 0;
  }
  // entries in table order: [start, start + width), width > 0
  DCB_HD void entry(uint32_t start, uint32_t width) {
    if (width > 16u) end_wide = start + width;
    if (start == 0) return;
    for (int j = 0; j < 6; ++j) {
      const uint32_t k = scale(j);
      if ((start & ((1u << k) - 1u)) == 0) continue;  // on a bucket edge: inside none
      const uint32_t bucket = start >> k;
      if (bucket == prev_bucket[j] && bad_at[j] == 0xFFFFFFFFu) bad_at[j] = start;
      prev_bucket[j] = bucket;
    }
  }
  // the cuts for wide-region buckets of 2^ka slots; false: the table does not have the shape
  DCB_HD bool cuts(uint32_t prec, uint32_t ka, uint32_t &ta, uint32_t &tb, uint32_t &tc) const {
    // 8-slot records cost what the byte region costs per slot, without its bitmap: they reach as far as they are good
    tc = bad_at[0] < prec ? bad_at[0] : prec;
    if (tc < end_wide) return false;
    tb = bad_at[1] < tc ? bad_at[1] : tc;
    const uint32_t fa = bad_at[ka - DCB_REC_KA0 + 2];
    ta = fa < tb ? fa : tb;
    return true;
  }
};

// ---- launch plan for the lane-per-stream rANS kernels ----
struct RansLaunch {
  StreamDesc *d_streams;          // device array of all streams of the shard
  const uint32_t *d_order;        // stream indices handled by this launch (sorted by length, desc)
  uint32_t n_streams;
  uint32_t lanes_per_warp;        // active lanes per warp-CTA
  uint32_t lut_bytes;             // per lane: LUT size (power of two)
  uint32_t lutb_bytes;            // per lane: narrow region of the two-region LUT (0 = uniform LUT only)
  uint32_t ent_bytes;             // per lane: cum[cap + 2] (+ val[cap_exc] for compact tables)
  uint32_t cap_entries;           // table entries a lane can hold
  uint32_t cap_exc;               // compact tables: entries beyond the dense prefix that need a value slot
  uint32_t lut_shift;             // log2(slots per LUT bucket)
  uint32_t prec_bits;             // rANS precision of the group
  uint32_t dump;                  // DCB_DUMP_* flags
  uint32_t compact;               // 1: tables indexed by active-symbol rank (+ value map), 0: by symbol id
  uint32_t zig;                   // symbols are zig-zag coded corrections
  uint32_t mode;                  // 0 generic post-processing, 1..4 specialised (dcb_device.cuh)
  uint32_t pairs;                 // chain/consumer warp pairs per CTA (dcb_rans_pc.cu); 0 = the single-warp kernels
  uint32_t direct;                // 1: direct slot LUT (lut_bytes = 6 << prec_bits per lane; warp-pair kernels only)
  uint32_t rec_ka;                // bucket-record kernels: log2(slots per record) of the wide region (0 = not that path)
  uint32_t rec_bytes;             // bucket-record kernels: table area per lane (records + byte region + bitmap + value map)
  uint32_t split;                 // warp-pair kernels: chain warps on sub-partitions 0..2, all consumers on sub-partition 3
};
