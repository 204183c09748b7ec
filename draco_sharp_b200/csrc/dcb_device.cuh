// draco_sharp_b200/csrc/dcb_device.cuh -- device helpers shared by the sm_100a kernels.
//
// Reference semantics restated here (src/Draco/IO/...):
//   zig-zag            BitUtilities.cs:72-81
//   wrap transform     Attributes/PredictionSchemes/PredictionSchemeWrapDecodingTransform.cs:46-67,
//                      PredictionSchemeWrapTransform.cs:67-100
//   octahedron xform   PredictionSchemeNormalOctahedron{,Canonicalized}DecodingTransform.cs,
//                      PredictionSchemeNormalOctahedronCanonicalizedTransform.cs:43-89, OctahedronToolBox.cs:144-212
//   dequantise         Attributes/AttributeQuantizationTransform.cs:179-199, Core/Dequantizer.cs:14-23
//   oct -> unit vector Attributes/AttributeOctahedronTransform.cs:82-102, OctahedronToolBox.cs:139-142,220-239
//   narrowing store    Attributes/SequentialIntegerAttributeDecoder.cs:142-160
// Float results are bit-exact with the C# evaluation order: every binary32 operation is rounded
// separately (explicit *_rn intrinsics, never contracted to FMA).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dcb_internal.h"
#include "dcb_kernels.h"

namespace dcb {

__device__ __forceinline__ int32_t zigzag_dec(uint32_t v) {
  // (v & 1) ? -(v >> 1) - 1 : v >> 1
  return (int32_t)((v >> 1) ^ (0u - (v & 1u)));
}

__device__ __forceinline__ int32_t wrap_original(int32_t pred, int32_t corr, int32_t mn, int32_t mx, int32_t max_diff) {
  pred = pred > mx ? mx : (pred < mn ? mn : pred);
  int32_t o = (int32_t)((uint32_t)pred + (uint32_t)corr);
  if (o > mx)
    o = (int32_t)((uint32_t)o - (uint32_t)max_diff);
  else if (o < mn)
    o = (int32_t)((uint32_t)o + (uint32_t)max_diff);
  return o;
}

// wrap_original for a REGULAR stream: the prediction is known to lie in [mn, mx] (every correction the stream's table can
// produce is smaller than max_diff in magnitude, so one +-max_diff always re-enters the range and the clamp of
// ClampPredictedValue, PredictionSchemeWrapTransformBase.cs, is the identity).  Same operations in the same order.
__device__ __forceinline__ int32_t wrap_regular(int32_t pred, int32_t corr, int32_t mn, int32_t mx, int32_t max_diff) {
  int32_t o = (int32_t)((uint32_t)pred + (uint32_t)corr);
  if (o > mx)
    o = (int32_t)((uint32_t)o - (uint32_t)max_diff);
  else if (o < mn)
    o = (int32_t)((uint32_t)o + (uint32_t)max_diff);
  return o;
}

struct OctBox {
  int32_t max_q, max_value, center;
  __device__ __forceinline__ void set(int bits) {
    max_q = (int32_t)((1u << bits) - 1u);
    max_value = max_q - 1;
    center = max_value / 2;
  }
};
__device__ __forceinline__ int32_t neg32(int32_t v) { return (int32_t)(0u - (uint32_t)v); }
__device__ __forceinline__ int32_t abs32(int32_t v) { return v < 0 ? neg32(v) : v; }
__device__ __forceinline__ bool oct_in_diamond(const OctBox &t, int32_t s, int32_t u) {
  return (uint32_t)abs32(s) + (uint32_t)abs32(u) <= (uint32_t)t.center;
}
// The octahedron helpers are written as straight-line select code: every lane of a warp decodes a different
// stream, so any data-dependent branch here would be divergent on almost every entry.
__device__ __forceinline__ void oct_invert_diamond(const OctBox &t, int32_t &s, int32_t &u) {
  const bool a = (s >= 0) & (u >= 0);
  const bool b = (s <= 0) & (u <= 0);
  const int32_t ss = a ? 1 : (b ? -1 : (s > 0 ? 1 : -1));
  const int32_t su = a ? 1 : (b ? -1 : (u > 0 ? 1 : -1));
  const int32_t cs = ss > 0 ? t.center : neg32(t.center), cu = su > 0 ? t.center : neg32(t.center);
  const int32_t us0 = (int32_t)((uint32_t)s + (uint32_t)s - (uint32_t)cs);
  const int32_t uu0 = (int32_t)((uint32_t)u + (uint32_t)u - (uint32_t)cu);
  const bool same = (ss == su);  // ss * su >= 0
  int32_t us = same ? neg32(uu0) : uu0;
  int32_t uu = same ? neg32(us0) : us0;
  us = (int32_t)((uint32_t)us + (uint32_t)cs);
  uu = (int32_t)((uint32_t)uu + (uint32_t)cu);
  s = us / 2;  // truncating, as C#
  u = uu / 2;
}
__device__ __forceinline__ int32_t oct_mod_max(const OctBox &t, int32_t x) {
  const int32_t hi = (int32_t)((uint32_t)x - (uint32_t)t.max_q);
  const int32_t lo = (int32_t)((uint32_t)x + (uint32_t)t.max_q);
  return x > t.center ? hi : (x < -t.center ? lo : x);
}
__device__ __forceinline__ void oct_rotate(int32_t &a, int32_t &b, int rot) {
  const int32_t x = a, y = b, nx = neg32(a), ny = neg32(b);
  a = rot == 1 ? y : (rot == 2 ? nx : (rot == 3 ? ny : x));
  b = rot == 1 ? nx : (rot == 2 ? ny : (rot == 3 ? x : y));
}
// pred (p0io,p1io) + correction (c0,c1) -> original, in place
__device__ __forceinline__ void oct_original(const OctBox &t, bool canonical, int32_t &p0io, int32_t &p1io,
                                             int32_t c0, int32_t c1) {
  int32_t p0 = (int32_t)((uint32_t)p0io - (uint32_t)t.center);
  int32_t p1 = (int32_t)((uint32_t)p1io - (uint32_t)t.center);
  const bool in_diamond = oct_in_diamond(t, p0, p1);
  {
    int32_t q0 = p0, q1 = p1;
    oct_invert_diamond(t, q0, q1);
    p0 = in_diamond ? p0 : q0;
    p1 = in_diamond ? p1 : q1;
  }
  // canonicalized transform: rotate the prediction into the bottom-left quadrant
  const bool bottom_left = ((p0 == 0) & (p1 == 0)) | ((p0 < 0) & (p1 <= 0));
  int rot = p0 == 0 ? (p1 == 0 ? 0 : (p1 > 0 ? 3 : 1)) : (p0 > 0 ? (p1 >= 0 ? 2 : 1) : (p1 <= 0 ? 0 : 3));
  rot = (canonical && !bottom_left) ? rot : 0;
  oct_rotate(p0, p1, rot);
  int32_t o0 = oct_mod_max(t, (int32_t)((uint32_t)p0 + (uint32_t)c0));
  int32_t o1 = oct_mod_max(t, (int32_t)((uint32_t)p1 + (uint32_t)c1));
  oct_rotate(o0, o1, (4 - rot) & 3);
  {
    int32_t q0 = o0, q1 = o1;
    oct_invert_diamond(t, q0, q1);
    o0 = in_diamond ? o0 : q0;
    o1 = in_diamond ? o1 : q1;
  }
  p0io = (int32_t)((uint32_t)o0 + (uint32_t)t.center);
  p1io = (int32_t)((uint32_t)o1 + (uint32_t)t.center);
}

// oct (s,t) -> unit vector; arithmetic types as the C# (binary32 coords and norm, binary64 1/sqrt and products)
__device__ __forceinline__ void oct_to_unit(int32_t s, int32_t u, float scale, float &ox, float &oy, float &oz) {
  float y = __fsub_rn(__fmul_rn(__int2float_rn(s), scale), 1.0f);
  float z = __fsub_rn(__fmul_rn(__int2float_rn(u), scale), 1.0f);
  const float x = __fsub_rn(__fsub_rn(1.0f, fabsf(y)), fabsf(z));
  const float x_offset = (-x < 0.0f) ? 0.0f : -x;
  y = __fadd_rn(y, (y < 0.0f) ? x_offset : -x_offset);
  z = __fadd_rn(z, (z < 0.0f) ? x_offset : -x_offset);
  const float ns = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
  if ((double)ns < 1E-6) {
    ox = 0.0f; oy = 0.0f; oz = 0.0f;
  } else {
    const double d = __ddiv_rn(1.0, __dsqrt_rn((double)ns));
    ox = __double2float_rn(__dmul_rn((double)x, d));
    oy = __double2float_rn(__dmul_rn((double)y, d));
    oz = __double2float_rn(__dmul_rn((double)z, d));
  }
}

// Per-stream constants of the reconstruction + store stages, loaded once per lane.
struct PostParams {
  int32_t recon, store, mn, mx, max_diff, dsize;
  bool zig;
  float qmin[4];
  float delta, oct_scale;
  OctBox box;
  __device__ void load(const StreamDesc &d) {
    recon = d.recon;
    store = d.store;
    zig = d.zigzag != 0;
    mn = d.xf_a;
    mx = d.xf_b;
    max_diff = (int32_t)(1u + (uint32_t)mx - (uint32_t)mn);
    box.set(2);
    delta = 0.0f;
    oct_scale = 0.0f;
    dsize = 4;
#pragma unroll
    for (int c = 0; c < 4; ++c) qmin[c] = 0.0f;
    if (recon == RECON_DELTA_OCT || recon == RECON_DELTA_OCT_CANON)
      box.set(32 - __clz(d.xf_a));  // bits = msb(max_q) + 1 (PredictionSchemeNormalOctahedronTransform.cs:44-53)
    if (store == STORE_DEQUANT) {
      const int32_t maxq = (int32_t)((1u << d.q_bits) - 1u);
      delta = __fdiv_rn(d.q_range, __int2float_rn(maxq));  // Dequantizer.cs:17
#pragma unroll
      for (int c = 0; c < 4; ++c) qmin[c] = d.q_min[c];
    } else if (store == STORE_OCT_UNIT) {
      const int32_t max_value = (int32_t)((1u << d.q_bits) - 2u);
      oct_scale = __fdiv_rn(2.0f, __int2float_rn(max_value));  // OctahedronToolBox.cs:19
    } else {
      dsize = dcb_dtype_len(d.data_type);
    }
  }
  // words of output per entry group of 4 entries
  __device__ __forceinline__ float dequant(int32_t q, int c) const {
    return __fadd_rn(__fmul_rn(__int2float_rn(q), delta), qmin[c]);
  }
};

// Store ONE entry (NCP portable ints in v) at entry index e of the attribute output.
template <int NCP>
__device__ __forceinline__ void store_entry(const PostParams &pp, int store, int dsize, uint8_t *optr, uint64_t e,
                                            const int32_t *v) {
  if (store == STORE_DEQUANT) {
    float *o = reinterpret_cast<float *>(optr) + e * NCP;
#pragma unroll
    for (int c = 0; c < NCP; ++c) o[c] = pp.dequant(v[c], c);
  } else if (store == STORE_OCT_UNIT) {
    if (NCP == 2) {
      float ox, oy, oz;
      oct_to_unit(v[0], v[NCP - 1], pp.oct_scale, ox, oy, oz);
      float *o = reinterpret_cast<float *>(optr) + e * 3;
      o[0] = ox; o[1] = oy; o[2] = oz;
    }
  } else {
    if (dsize == 1) {
      uint8_t *o = optr + e * NCP;
#pragma unroll
      for (int c = 0; c < NCP; ++c) o[c] = (uint8_t)v[c];
    } else if (dsize == 2) {
      uint16_t *o = reinterpret_cast<uint16_t *>(optr) + e * NCP;
#pragma unroll
      for (int c = 0; c < NCP; ++c) o[c] = (uint16_t)v[c];
    } else {
      int32_t *o = reinterpret_cast<int32_t *>(optr) + e * NCP;
#pragma unroll
      for (int c = 0; c < NCP; ++c) o[c] = v[c];
    }
  }
}

// Store a GROUP of 4 consecutive entries starting at entry index e4 (a multiple of 4): the group
// occupies 4 * bytes_per_entry bytes starting on a 16-byte boundary whenever that size is a multiple
// of 16 (attribute outputs start on 128-byte boundaries), so it is written as 128-bit stores.
template <int NCP>
__device__ __forceinline__ void store_group4(const PostParams &pp, int store, int dsize, uint8_t *optr, uint64_t e4,
                                             const int32_t (*v)[NCP]) {
  if (store == STORE_DEQUANT) {
    float f[4 * NCP];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int c = 0; c < NCP; ++c) f[j * NCP + c] = pp.dequant(v[j][c], c);
    float4 *o = reinterpret_cast<float4 *>(reinterpret_cast<float *>(optr) + e4 * NCP);
#pragma unroll
    for (int k = 0; k < NCP; ++k) o[k] = make_float4(f[4 * k], f[4 * k + 1], f[4 * k + 2], f[4 * k + 3]);
  } else if (store == STORE_OCT_UNIT) {
    if (NCP == 2) {
      float f[12];
#pragma unroll
      for (int j = 0; j < 4; ++j) oct_to_unit(v[j][0], v[j][NCP - 1], pp.oct_scale, f[3 * j], f[3 * j + 1], f[3 * j + 2]);
      float4 *o = reinterpret_cast<float4 *>(reinterpret_cast<float *>(optr) + e4 * 3);
#pragma unroll
      for (int k = 0; k < 3; ++k) o[k] = make_float4(f[4 * k], f[4 * k + 1], f[4 * k + 2], f[4 * k + 3]);
    }
  } else if (dsize == 4) {
    int4 *o = reinterpret_cast<int4 *>(reinterpret_cast<int32_t *>(optr) + e4 * NCP);
    const int32_t *f = &v[0][0];
#pragma unroll
    for (int k = 0; k < NCP; ++k) o[k] = make_int4(f[4 * k], f[4 * k + 1], f[4 * k + 2], f[4 * k + 3]);
  } else if (dsize == 1) {
    // 4 entries x NCP bytes = NCP 32-bit words
    uint32_t *o = reinterpret_cast<uint32_t *>(optr + e4 * NCP);
    const int32_t *f = &v[0][0];
#pragma unroll
    for (int k = 0; k < NCP; ++k)
      o[k] = ((uint32_t)f[4 * k] & 0xFFu) | (((uint32_t)f[4 * k + 1] & 0xFFu) << 8) |
             (((uint32_t)f[4 * k + 2] & 0xFFu) << 16) | (((uint32_t)f[4 * k + 3] & 0xFFu) << 24);
  } else {
    // 4 entries x NCP x 2 bytes = 2 * NCP 32-bit words
    uint32_t *o = reinterpret_cast<uint32_t *>(optr + e4 * NCP * 2);
    const int32_t *f = &v[0][0];
#pragma unroll
    for (int k = 0; k < 2 * NCP; ++k) o[k] = ((uint32_t)f[2 * k] & 0xFFFFu) | (((uint32_t)f[2 * k + 1] & 0xFFFFu) << 16);
  }
}

// ---------------------------------------------------------------------------------------------
// rANS lane: everything one lane needs to run one stream's chain.
//
// Shared-memory layout of a warp-CTA (all regions sized for `lanes` lanes, uniform per launch):
//   LUT region     lane l at  lut0 + l * lut_bytes        lut_bytes = nb * sizeof(T), power of two, region
//                                                          aligned to lut_bytes  ->  address = base | index
//   ring region    lane l at  ring0 + l * 128             128-byte aligned       ->  address = base | offset
//   entry region   lane l at  ent0 + l * ent_bytes        cum[ne + 2] then val[ne] (T each)
// LUT entries hold the byte offset (from ent0) of cum[i] for the first table entry i that owns part
// of the bucket, so the second-level loads need no index arithmetic.  T = uint16_t needs 2^prec and
// lanes * ent_bytes below 65536, else uint32_t.
//
// compressed bytes: rANS consumes the payload from its END towards its start (RAnsDecoder.cs:60
// `Buffer[--BufferOffset]`).  Every lane owns a 128-byte ring, direct-mapped by arena address (byte g
// lives at ring[g % 128]); 16-byte chunks are pulled ahead of the read position with per-lane
// cp.async (LDGSTS), so the per-symbol byte fetch is two aligned LDS + one funnel shift.
// ---------------------------------------------------------------------------------------------
#ifndef DCB_RING_BYTES
#define DCB_RING_BYTES 128u
#endif

__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void *gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(smem_addr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(a));
  return v;
}

// geometry of the tables of one launch (uniform over the grid)
struct TableGeom {
  uint32_t lut_bytes;   // per lane, power of two (uniform LUT / wide region of the two-region LUT)
  uint32_t lutb_bytes;  // per lane: narrow region of the two-region LUT (one byte per 2 slots), 0 = none
  uint32_t blk_bytes;   // per lane: block bases of the narrow region (one u32 per 128 slots), power of two
  uint32_t ent_bytes;   // per lane
  uint32_t cap_entries; // table entries a lane can hold
  uint32_t cap_exc;     // compact tables: value slots for entries beyond the dense symbol prefix
  uint32_t lut_shift;   // log2(slots per LUT bucket)
  uint32_t compact;     // 1: entries = symbols with prob > 0 (+ value map), 0: entries = symbol ids
  uint32_t zig;         // value map holds zig-zag decoded values (compact) / apply zig-zag (dense)
  uint32_t direct_prec; // rANS precision of the launch (direct slot LUT geometry)
  uint32_t direct;      // 1: direct slot LUT (three u16 arrays of 2^prec slots per lane: freq | offset | entry), lut_bytes = 6 << prec
};

template <typename T, bool GLOBAL>
struct RansLane {
  // state chain
  uint32_t x;
  uint32_t p1;          // low 32 bits of (arena offset of the next unread byte) = ptr - 1
  // constants
  uint32_t L, L8, L16, mask, prec_bits;
  uint32_t lut_base;    // smem address (GLOBAL: byte offset) of the lane's LUT
  uint32_t lut_mask, lut_sh;
  uint32_t ring;        // smem address of the lane's ring
  uint32_t ent_off;     // byte offset of the lane's cum[0] from ent0
  uint32_t val_delta;   // byte distance cum[i] -> its value slot (entries beyond the dense prefix)
  uint32_t dprefix;     // compact tables: entries 0..dprefix-1 are the symbols 0..dprefix-1
  // two-region LUT (u16 tables in shared memory): slots below t_split are bucketed by 2^kA, where every table
  // entry is at least 2^kA slots wide; slots from t_split on are bucketed by 2.  Either way a bucket meets at
  // most two entries, so the probe needs no search loop.
  // Region A holds u16 entry ranks.  Region B holds, per 2-slot bucket, a u8 rank relative to the first entry
  // of its 128-slot block, and per block the shared-memory address of that entry's cum value.
  uint32_t t_split, a_sh, a_mask, b_base, base_b;
  uint32_t lutb_addr;   // smem address of the lane's region B deltas
  uint32_t blk_addr;    // smem address of the lane's block bases (aligned to blk_bytes)
  uint32_t blk_mask;
  uint32_t cum_addr;    // smem address of the lane's cum[0]
  uint32_t n_entries_tab;  // entries built (ne)
  bool split_ok;        // the two-region LUT fits this lane's LUT capacity
  uint32_t max_abs_val; // largest magnitude a zig-zag decoded symbol of this table can have (lean main loop: regular streams)
  // direct slot LUT (low-residency launches): shared-memory addresses of the lane's freq[], offset[] and entry[] arrays
  // (u16 per slot).  One dependent LDS per symbol instead of two: x' = q * freq[r] + offset[r] (RAnsDecoder.cs:90-99
  // with lut[] / prob[] / cum[] folded per slot, which is what BuildLookupTable :69-88 itself materialises).
  uint32_t d_freq, d_off, d_ent;
  const uint8_t *ent0;  // entry region (generic pointer: shared or global)
  const uint8_t *lut0;  // GLOBAL only
  // byte supply: the payload is requested into the ring downwards from its end rounded up to 16 bytes
  const uint8_t *lo_ptr;  // lowest byte requested so far
  uint32_t lo;            // low 32 bits of its arena offset (a multiple of 16)
  uint32_t p1_init;
  uint32_t off_init;      // unread payload bytes at init (BufferOffset)

  __device__ __forceinline__ uint32_t consumed() const { return p1_init - p1; }
  __device__ __forceinline__ uint32_t bytes_left() const { return off_init - consumed(); }

  // Requests the 16-byte chunks that keep the ring filled down to 128 bytes below the read position (at most
  // MAX_CHUNKS of them) and commits them as one group.  The chunk count comes from one 32-bit distance, every chunk has
  // a predicate of its own and its source is a fixed offset from lo_ptr: no branch and no 64-bit compare chain (the main
  // loops call this once per 4 entries).
  template <int MAX_CHUNKS>
  __device__ __forceinline__ void top_up() {
    const uint32_t floor_lo = ((p1 + 16u) & ~15u) - DCB_RING_BYTES;  // never above lo
    const uint32_t n = min((lo - floor_lo) >> 4, (uint32_t)MAX_CHUNKS);
#pragma unroll
    for (int k = 0; k < MAX_CHUNKS; ++k) {
      asm volatile("{\n .reg .pred p;\n setp.gt.u32 p, %2, %3;\n @p cp.async.ca.shared.global [%0], [%1], 16;\n}\n"
                   ::"r"(ring | ((lo - 16u * (k + 1)) & (DCB_RING_BYTES - 1u))), "l"(lo_ptr - 16 * (k + 1)), "r"(n),
                   "r"((uint32_t)k) : "memory");
    }
    lo -= n << 4;
    lo_ptr -= n << 4;
    cp_async_commit();
  }

  // the 4 bytes [ptr-4, ptr) with byte ptr-1 in the most significant position: the two ring words are
  // requested as soon as the read position is known (prefetch), combined when the next step needs them
  uint32_t pk_hi, pk_lo, pk_sh;
  __device__ __forceinline__ void prefetch() {
    pk_hi = lds_u32(ring | (p1 & (DCB_RING_BYTES - 4u)));
    pk_lo = lds_u32(ring | ((p1 + DCB_RING_BYTES - 4u) & (DCB_RING_BYTES - 4u)));
    pk_sh = (p1 & 3u) * 8u + 8u;
  }
  __device__ __forceinline__ uint32_t peek() const { return __funnelshift_rc(pk_lo, pk_hi, pk_sh); }

  __device__ __forceinline__ uint32_t lut_load(uint32_t xx) const {
    const uint32_t a = lut_base | ((xx >> lut_sh) & lut_mask);
    if (GLOBAL) return *reinterpret_cast<const T *>(lut0 + a);
    uint32_t v;
    if (sizeof(T) == 2) asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(v) : "r"(a));
    else asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(a));
    return v;
  }

  // One RAnsDecoder.Read() (RAnsDecoder.cs:56-67,90-99): renormalise, then decode.
  //   while (state < L && off > 0) state = state * 256 + buf[--off];
  // L is a multiple of 256, so the iteration count depends on x alone: one per threshold L, L/256,
  // L/65536 that x is below, capped by the bytes left.  CAREFUL = false assumes the caller has
  // checked that enough bytes are left for the cap not to bind.
  // Returns the byte offset (from ent0) of cum[entry].
  // PROBE: 0 uniform LUT (+ rare search), 1 two-region LUT, 2 direct slot LUT
  template <bool CAREFUL, int PROBE>
  __device__ __forceinline__ uint32_t step() {
    const uint32_t v = peek();
    uint32_t sh;  // 8 * bytes to shift in
    if (sizeof(T) == 2 && !GLOBAL) {
      // precision <= 15: x >= 4 > L/65536, at most two bytes
      const uint32_t sh2 = x < L8 ? 16u : 8u;
      sh = x < L ? sh2 : 0u;
    } else {
      const uint32_t sh3 = x < L16 ? 24u : 16u;
      const uint32_t sh2 = x < L8 ? sh3 : 8u;
      sh = x < L ? sh2 : 0u;
    }
    if (CAREFUL) sh = min(sh, 8u * bytes_left());
    const uint32_t xr = __funnelshift_l(v, x, sh);
    p1 -= sh >> 3;
    prefetch();
    const uint32_t r = xr & mask;
    const uint32_t q = xr >> prec_bits;
    uint32_t o, c0, c1, c2;
    if (PROBE == 2) {
      const uint32_t r2 = r << 1;
      uint32_t f, off;
      asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(f) : "r"(d_freq + r2));
      asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(off) : "r"(d_off + r2));
      asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(o) : "r"(d_ent + r2));  // off the chain: only the value map wants it
      x = q * f + off;
      return o;
    }
    if (PROBE == 1) {
      // both regions hold u8 ranks relative to the first entry of their 128-slot block; blk[] holds the
      // shared-memory address of that entry's cum value: one byte load + one word load, issued together
      const uint32_t a_a = ((xr >> a_sh) & a_mask) | lut_base;
      const uint32_t a_b = (r >> 1) + b_base;
      const uint32_t a = r >= t_split ? a_b : a_a;
      const uint32_t a_k = ((xr >> 5) & blk_mask) | blk_addr;
      uint32_t dl, bb;
      asm volatile("ld.shared.u8 %0, [%1];\n" : "=r"(dl) : "r"(a));
      asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(bb) : "r"(a_k));
      const uint32_t ca = dl * 2u + bb;
      asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(c0) : "r"(ca));
      asm volatile("ld.shared.u16 %0, [%1+2];\n" : "=r"(c1) : "r"(ca));
      asm volatile("ld.shared.u16 %0, [%1+4];\n" : "=r"(c2) : "r"(ca));
      const uint32_t rank = (ca - cum_addr) >> 1;
      o = ent_off + 2u * rank;
    } else {
      o = lut_load(xr);
      const T *cp = reinterpret_cast<const T *>(ent0 + o);
      c0 = cp[0];
      c1 = cp[1];
      c2 = cp[2];
      // uniform LUT: a bucket may meet three or more entries (rare by construction of the granularity)
      if (__builtin_expect(r >= c2, 0)) {
        do {
          o += (uint32_t)sizeof(T);
          c0 = c1;
          c1 = c2;
          c2 = *reinterpret_cast<const T *>(ent0 + o + 2u * (uint32_t)sizeof(T));
        } while (r >= c2);
      }
    }
    const bool second = r >= c1;
    const uint32_t xa = q * (c1 - c0) + (r - c0);
    const uint32_t xb = q * (c2 - c1) + (r - c1);
    x = second ? xb : xa;
    return o + (second ? (uint32_t)sizeof(T) : 0u);
  }

  // direct slot LUT, main loop: returns the SLOT; the consumer warp looks the table entry up (d_ent[slot])
  __device__ __forceinline__ uint32_t step_direct_slot() {
    const uint32_t v = peek();
    const uint32_t sh2 = x < L8 ? 16u : 8u;  // u16 tables: precision <= 15, at most two bytes (see step)
    const uint32_t sh = x < L ? sh2 : 0u;
    const uint32_t xr = __funnelshift_l(v, x, sh);
    p1 -= sh >> 3;
    prefetch();
    const uint32_t r = xr & mask;
    const uint32_t q = xr >> prec_bits;
    const uint32_t r2 = r << 1;
    uint32_t f, off;
    asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(f) : "r"(d_freq + r2));
    asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(off) : "r"(d_off + r2));
    x = q * f + off;
    return r;
  }

  // ---- lean main loop (u16 tables in shared memory, two-region LUT) ----
  // Byte window: the 8 payload bytes below the read position, newest byte in the top bits of w_hi.  Three symbols of a
  // u16 table consume at most 6 bytes, so the window is opened once per three symbols (three aligned ring words, two
  // funnel shifts) instead of two ring words + shift bookkeeping per symbol.
  uint32_t w_hi, w_lo, w_cb;
  __device__ __forceinline__ void window_open() {
    const uint32_t W0 = lds_u32(ring | (p1 & (DCB_RING_BYTES - 4u)));
    const uint32_t W1 = lds_u32(ring | ((p1 + DCB_RING_BYTES - 4u) & (DCB_RING_BYTES - 4u)));
    const uint32_t W2 = lds_u32(ring | ((p1 + DCB_RING_BYTES - 8u) & (DCB_RING_BYTES - 4u)));
    const uint32_t sh = (p1 & 3u) * 8u + 8u;
    w_hi = __funnelshift_rc(W1, W0, sh);
    w_lo = __funnelshift_rc(W2, W1, sh);
    w_cb = 0;
  }
  __device__ __forceinline__ void window_close() { p1 -= w_cb >> 3; }
  // One RAnsDecoder.Read() inside an open window; the caller has checked that the bytes cannot run out.  Same probe as
  // step<false, 1>; the renormalisation is two predicated funnel shifts (RAnsDecoder.cs:58-61, at most two bytes for
  // precision <= 15).  Returns the shared-memory ADDRESS of cum[entry].
  // GATED: the rank-byte load is predicated on (gate & zero) == 0 with `zero` a register the compiler cannot see through
  // (always true at run time).  It ties the load to the instructions that produce `gate` -- the post-processing of an
  // EARLIER symbol -- so that ptxas has to place that work before this step's table probe instead of clumping it at the
  // end of the unrolled group (software-pipelined main loop, run_stream_lean_sp).
  template <bool FIRST, bool GATED = false>
  __device__ __forceinline__ uint32_t step_lean(uint32_t gate = 0u, uint32_t zero = 0u) {
    const uint32_t v = FIRST ? w_hi : __funnelshift_lc(w_lo, w_hi, w_cb);
    const bool one = x < L, two = x < L8;
    uint32_t xr = x;
    if (one) xr = __funnelshift_l(v, x, 8);
    if (two) xr = __funnelshift_l(v, x, 16);
    if (FIRST) w_cb = one ? 8u : 0u;
    else if (one) w_cb += 8u;
    if (two) w_cb += 8u;
    const uint32_t r = xr & mask;
    const uint32_t q = xr >> prec_bits;
    const uint32_t a_a = ((xr >> a_sh) & a_mask) | lut_base;
    const uint32_t a_b = (r >> 1) + b_base;
    const uint32_t a = r >= t_split ? a_b : a_a;
    const uint32_t a_k = ((xr >> 5) & blk_mask) | blk_addr;
    uint32_t dl, bb, c0, c1, c2;
    if (GATED)
      asm volatile("{\n .reg .pred p;\n .reg .b32 t;\n and.b32 t, %2, %3;\n setp.eq.u32 p, t, 0;\n @p ld.shared.u8 %0, [%1];\n}\n"
                   : "=r"(dl) : "r"(a), "r"(gate), "r"(zero));
    else
      asm volatile("ld.shared.u8 %0, [%1];\n" : "=r"(dl) : "r"(a));
    asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(bb) : "r"(a_k));
    const uint32_t ca = dl * 2u + bb;
    // one block: ptxas has been seen to issue the third load only after the first two came back (a third LDS latency)
    asm volatile("ld.shared.u16 %1, [%3+2];\n ld.shared.u16 %2, [%3+4];\n ld.shared.u16 %0, [%3];\n"
                 : "=r"(c0), "=r"(c1), "=r"(c2) : "r"(ca));
    const bool second = r >= c1;
    const uint32_t xa = q * (c1 - c0) + (r - c0);
    const uint32_t xb = q * (c2 - c1) + (r - c1);
    x = second ? xb : xa;
    return ca + (second ? 2u : 0u);
  }
  // The same inside the direct slot LUT (low-residency launches): ONE dependent access per symbol.  Returns the
  // shared-memory address of cum[entry] like step_lean (the entry[] load is off the chain: only the value map wants it).
  template <bool FIRST>
  __device__ __forceinline__ uint32_t step_lean_direct(uint32_t gate, uint32_t zero) {
    const uint32_t v = FIRST ? w_hi : __funnelshift_lc(w_lo, w_hi, w_cb);
    const bool one = x < L, two = x < L8;
    uint32_t xr = x;
    if (one) xr = __funnelshift_l(v, x, 8);
    if (two) xr = __funnelshift_l(v, x, 16);
    if (FIRST) w_cb = one ? 8u : 0u;
    else if (one) w_cb += 8u;
    if (two) w_cb += 8u;
    const uint32_t r2 = (xr & mask) << 1;
    const uint32_t q = xr >> prec_bits;
    uint32_t f, off, o;
    asm volatile(
        "{\n .reg .pred p;\n .reg .b32 t;\n and.b32 t, %6, %7;\n setp.eq.u32 p, t, 0;\n"
        " @p ld.shared.u16 %0, [%3];\n @p ld.shared.u16 %1, [%4];\n @p ld.shared.u16 %2, [%5];\n}\n"
        : "=r"(f), "=r"(off), "=r"(o)
        : "r"(d_freq + r2), "r"(d_off + r2), "r"(d_ent + r2), "r"(gate), "r"(zero));
    x = q * f + off;
    return o + (cum_addr - ent_off);
  }
  // value of the entry whose cum lives at shared-memory address ca (compact u16 tables, zig-zag decoded value slots)
  __device__ __forceinline__ int32_t value_at(uint32_t ca) const {
    const uint32_t rank2 = ca - cum_addr;  // 2 * rank
    if (rank2 >= 2u * dprefix) {
      int32_t v;
      asm volatile("ld.shared.s16 %0, [%1];\n" : "=r"(v) : "r"(ca + val_delta));
      return v;
    }
    return zigzag_dec(rank2 >> 1);
  }

  // the same for symbols that are not zig-zag coded (tags): the value slots of a compact table hold symbol ids
  __device__ __forceinline__ uint32_t value_at_plain(uint32_t ca, bool compact) const {
    const uint32_t rank2 = ca - cum_addr;  // 2 * rank
    if (compact && rank2 >= 2u * dprefix) {
      uint32_t v;
      asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(v) : "r"(ca + val_delta));
      return v;
    }
    return rank2 >> 1;
  }

  // table entry -> symbol value.  dense: the entry index is the symbol id.  compact: entries below the dense
  // prefix are their own symbol ids, the others carry a value slot (zig-zag decoded when zig).
  __device__ __forceinline__ int32_t value(uint32_t o, bool compact, bool zig) const {
    const uint32_t rank = (o - ent_off) / (uint32_t)sizeof(T);
    if (compact && rank >= dprefix) {
      if (sizeof(T) == 2) {
        return zig ? (int32_t) * reinterpret_cast<const int16_t *>(ent0 + o + val_delta)
                   : (int32_t) * reinterpret_cast<const uint16_t *>(ent0 + o + val_delta);
      }
      return *reinterpret_cast<const int32_t *>(ent0 + o + val_delta);
    }
    return zig ? zigzag_dec(rank) : (int32_t)rank;
  }
  // the symbol id itself (debug dumps)
  __device__ __forceinline__ uint32_t symbol(uint32_t o, const TableGeom &g) const {
    const int32_t v = value(o, g.compact != 0, g.zig != 0);
    if (!g.zig) return (uint32_t)v;
    return v >= 0 ? ((uint32_t)v << 1) : ((((uint32_t)(-(v + 1))) << 1) | 1u);
  }

  // RAnsDecoder.ReadInit (RAnsDecoder.cs:20-54)
  __device__ int init_state(const uint8_t *arena_, const StreamDesc &d) {
    const uint64_t n = d.payload_len;
    if (n < 1) return DCB_ERR_RANS_INIT;
    const uint8_t *p = arena_ + d.payload_off;
    const uint32_t tag = (uint32_t)p[n - 1] >> 6;
    if (n < tag + 1) return DCB_ERR_RANS_INIT;
    uint32_t v = 0;
    for (uint32_t i = 0; i <= tag; ++i) v |= (uint32_t)p[n - 1 - tag + i] << (8 * i);
    v &= (tag == 0) ? 0x3Fu : (tag == 1) ? 0x3FFFu : (tag == 2) ? 0x3FFFFFu : 0x3FFFFFFFu;
    prec_bits = d.prec_bits;
    L = 4u << d.prec_bits;
    L8 = L >> 8;
    L16 = L >> 16;
    mask = (1u << d.prec_bits) - 1u;
    x = v + L;
    if (x >= L * 256u) return DCB_ERR_RANS_INIT;
    off_init = (uint32_t)(n - (tag + 1));
    const uint64_t end = d.payload_off + off_init;  // arena offset one past the first unread byte
    p1_init = (uint32_t)end - 1u;
    p1 = p1_init;
    lo_ptr = arena_ + ((end + 15u) & ~15ull);
    lo = ((uint32_t)end + 15u) & ~15u;
    return DCB_OK;
  }
  __device__ __forceinline__ void init_ring(uint32_t ring_addr) {
    ring = ring_addr;
    top_up<DCB_RING_BYTES / 16>();
    cp_async_wait<0>();
    prefetch();
  }

  // Parse RANS_TABLE at d.table_off into the lane's cum / value arrays (RAnsSymbolDecoder.cs:12-51,
  // RAnsDecoder.cs:69-88) and decide whether the two-region LUT fits.  The LUT itself is written by fill_lut.
  __device__ int build(const uint8_t *arena_, const StreamDesc &d, const TableGeom &g, T *ent, uint32_t ent_off_) {
    ent_off = ent_off_;
    lut_sh = g.lut_shift - (sizeof(T) == 2 ? 1u : 2u);
    lut_mask = g.lut_bytes - (uint32_t)sizeof(T);
    split_ok = false;
    T *cum = ent;
    T *val = ent + g.cap_entries + 2u;   // value slot of entry (dprefix + j) is val[j]
    uint64_t pos = d.table_off;
    const uint64_t bend = d.buf_end;
    for (int i = 0; i < 10; ++i) {  // skip the num_symbols varint (value parsed by the indexer)
      if (pos >= bend) return DCB_ERR_EOF;
      if (!(arena_[pos++] & 0x80)) break;
    }
    const uint32_t ns = d.num_symbols;
    const uint32_t prec = 1u << d.prec_bits;
    if (!g.compact && ns > g.cap_entries) return DCB_ERR_TABLE;
    dprefix = g.compact ? 0xFFFFFFFFu : 0u;  // compact: set at the first entry whose symbol id != its rank
    uint64_t c = 0;
    uint32_t ne = 0;
    bool overflow = false;
    uint32_t last_sym = 0;  // largest symbol id with a non-zero probability
    for (uint32_t i = 0; i < ns; ++i) {
      if (pos >= bend) return DCB_ERR_EOF;
      const uint32_t pd = arena_[pos++];
      const uint32_t token = pd & 3u;
      if (token == 3u) {
        const uint32_t off = pd >> 2;
        if (i + off >= ns) return DCB_ERR_TABLE;
        if (!g.compact)
          for (uint32_t j = 0; j <= off; ++j) cum[i + j] = (T)(c > prec ? prec : c);
        i += off;
      } else {
        uint32_t prob = pd >> 2;
        for (uint32_t b = 0; b < token; ++b) {
          if (pos >= bend) return DCB_ERR_EOF;
          prob |= (uint32_t)arena_[pos++] << (8 * (b + 1) - 2);
        }
        if (prob) last_sym = i;
        if (g.compact) {
          if (prob) {
            if (c + prob > prec || ne >= g.cap_entries) overflow = true;
            if (!overflow) {
              if (dprefix == 0xFFFFFFFFu && i != ne) dprefix = ne;
              if (dprefix != 0xFFFFFFFFu) {
                if (ne - dprefix >= g.cap_exc) overflow = true;
                else val[ne - dprefix] = (T)(g.zig ? (uint32_t)zigzag_dec(i) : i);
              }
              if (!overflow) {
                cum[ne] = (T)c;
                ++ne;
              }
            }
          }
        } else {
          if (c + prob > prec) overflow = true;
          cum[i] = (T)(c > prec ? prec : c);
        }
        c += prob;
      }
    }
    if (overflow || c != prec) return DCB_ERR_TABLE;
    if (!g.compact) ne = ns;
    if (g.compact && dprefix == 0xFFFFFFFFu) dprefix = ne;
    cum[ne] = (T)prec;
    cum[ne + 1] = (T)prec;  // pad: the two-candidate probe reads cum[i + 2]
    n_entries_tab = ne;
    max_abs_val = (last_sym + 1u) >> 1;  // |zigzag_dec(i)| = (i + 1) / 2
    val_delta = (g.cap_entries + 2u - (g.compact ? dprefix : 0u)) * (uint32_t)sizeof(T);
    // ---- two-region LUT: pick the bucket size 2^kA of the wide region that needs the fewest LUT bytes ----
    // Dense tables may hold zero-width entries between two owners of one bucket (the two-candidate probe would
    // stop at the empty one), so the split LUT is only built for compact tables.
    if (sizeof(T) == 2 && !GLOBAL && g.compact && g.lutb_bytes > 0) {
      uint32_t first_narrow[8];  // first slot owned by an entry narrower than 2^kA (kA = 1..7)
#pragma unroll
      for (int k = 1; k <= 7; ++k) first_narrow[k] = prec;
      for (uint32_t i = 0; i < ne; ++i) {
        const uint32_t w = (uint32_t)cum[i + 1] - (uint32_t)cum[i];
#pragma unroll
        for (int k = 1; k <= 7; ++k)
          if (w < (1u << k) && first_narrow[k] == prec) first_narrow[k] = (uint32_t)cum[i];
      }
      uint32_t best = 0xFFFFFFFFu, best_k = 0, best_t = 0;
#pragma unroll
      for (int k = 1; k <= 7; ++k) {
        if ((uint32_t)k + 7u > d.prec_bits) continue;
        const uint32_t t = first_narrow[k] & ~127u;   // whole 128-slot blocks on either side
        const uint32_t na = t >> k, nbk = (prec - t) >> 1;
        if (na > g.lut_bytes || nbk > g.lutb_bytes) continue;
        const uint32_t need = na + nbk;
        if (need < best) { best = need; best_k = (uint32_t)k; best_t = t; }
      }
      if (best_k > 0 && g.blk_bytes >= ((prec >> 7) << 2)) {
        split_ok = true;
        t_split = best_t;
        a_sh = best_k;
        a_mask = (1u << (d.prec_bits - best_k)) - 1u;
        b_base = lutb_addr - (best_t >> 1);
        blk_mask = ((prec >> 7) - 1u) << 2;
      }
    }
    return DCB_OK;
  }

  // LUT entries: byte offset (from ent0) of cum[i] for the first table entry i owning part of the bucket
  __device__ void fill_lut(const TableGeom &g, T *lut, uint8_t *lutb, uint32_t *blk, const T *cum, bool split) const {
    const uint32_t prec = 1u << prec_bits;
    uint32_t i = 0;
    if (!split) {
      const uint32_t nb = prec >> g.lut_shift;
      for (uint32_t b = 0; b < nb; ++b) {
        const uint32_t slot = b << g.lut_shift;
        while ((uint32_t)cum[i + 1] <= slot) ++i;
        lut[b] = (T)(ent_off + i * (uint32_t)sizeof(T));
      }
      return;
    }
    const uint32_t ka = a_sh;
    const uint32_t na = t_split >> ka;
    uint8_t *luta = reinterpret_cast<uint8_t *>(lut);
    uint32_t cur_blk = 0xFFFFFFFFu, base_rank = 0;
    for (uint32_t b = 0; b < na; ++b) {
      const uint32_t slot = b << ka;
      while ((uint32_t)cum[i + 1] <= slot) ++i;
      if ((slot >> 7) != cur_blk) {  // first bucket of a 128-slot block: its owner is the block's base entry
        cur_blk = slot >> 7;
        base_rank = i;
        blk[cur_blk] = cum_addr + 2u * i;
      }
      luta[b] = (uint8_t)(i - base_rank);
    }
    const uint32_t nbk = (prec - t_split) >> 1;
    for (uint32_t b = 0; b < nbk; ++b) {
      const uint32_t slot = t_split + 2u * b;
      while ((uint32_t)cum[i + 1] <= slot) ++i;
      if ((slot >> 7) != cur_blk) {
        cur_blk = slot >> 7;
        base_rank = i;
        blk[cur_blk] = cum_addr + 2u * i;
      }
      lutb[b] = (uint8_t)(i - base_rank);
    }
  }
};

// ---------------------------------------------------------------------------------------------
// pieces shared by the lane-per-stream rANS kernels (dcb_kernels.cu, dcb_rans_pc.cu)
// ---------------------------------------------------------------------------------------------
// post-processing mode of a launch: 0 = per-stream (runtime) recon/store kinds; the others pin them at
// compile time for the hot shapes
//   1  delta + wrap  -> dequantise to float      (quantized positions / tex coords)
//   2  delta + wrap  -> narrow to uint8          (colours)
//   3  normals: the unsigned corrections go to the int32 scratch as they are; the octahedral recurrence is a chain of
//      its own (~120 dependent-ish instructions per entry) and runs in oct_chain_kernel, next to the rANS kernels of
//      the batch's other attributes instead of in front of them
//   4  parallelogram streams: zig-zag decoded corrections to the int32 scratch (para_chain_kernel does the rest)
template <int MODE>
__device__ __forceinline__ int recon_of(const PostParams &pp) {
  return (MODE == 1 || MODE == 2) ? (int)RECON_DELTA_WRAP : ((MODE == 3 || MODE == 4) ? (int)RECON_NONE : pp.recon);
}
template <int MODE>
__device__ __forceinline__ int store_of(const PostParams &pp) {
  // normals leave the serial kernels as quantized (s, t) pairs: the unit-vector conversion (double precision
  // 1/sqrt, as the C#) runs in oct_unit_kernel, point-parallel, instead of stretching the serial chain
  return MODE == 1 ? (int)STORE_DEQUANT : ((MODE == 2 || MODE == 3 || MODE == 4) ? (int)STORE_NARROW : pp.store);
}
template <int MODE>
__device__ __forceinline__ int dsize_of(const PostParams &pp) {
  return MODE == 2 ? 1 : ((MODE == 3 || MODE == 4) ? 4 : pp.dsize);
}

// shared-memory carve-up of a warp-CTA (see RansLane)
struct SmemLayout {
  uint32_t lut0, ring0, blk0, lutb0, ent0;  // byte offsets from the dynamic shared-memory base
};
__device__ __forceinline__ SmemLayout smem_layout(uint32_t base_addr, uint32_t lanes, const TableGeom &g, bool table_global) {
  SmemLayout l;
  uint32_t a = base_addr;
  if (!table_global) {
    if (g.direct) a = (a + 15u) & ~15u;
    else a = (a + g.lut_bytes - 1u) & ~(g.lut_bytes - 1u);
    l.lut0 = a - base_addr;
    a += lanes * g.lut_bytes;
  } else {
    l.lut0 = 0;
  }
  a = (a + DCB_RING_BYTES - 1u) & ~(DCB_RING_BYTES - 1u);
  l.ring0 = a - base_addr;
  a += lanes * DCB_RING_BYTES;
  l.blk0 = l.lutb0 = a - base_addr;
  if (!table_global && g.lutb_bytes) {
    a = (a + g.blk_bytes - 1u) & ~(g.blk_bytes - 1u);
    l.blk0 = a - base_addr;
    a += lanes * g.blk_bytes;
    l.lutb0 = a - base_addr;
    a += (lanes * g.lutb_bytes + 15u) & ~15u;
  }
  l.ent0 = a - base_addr;
  return l;
}

// decode one entry: NCP symbols -> corrections -> prediction; leaves the portable ints in v and prev
// TAB: 0 = table kind (dense / compact) read from the launch geometry, 1 = dense, 2 = compact
template <int NCP, typename T, bool TG, bool DUMP, int MODE, int TAB, bool CAREFUL, int PROBE>
__device__ __forceinline__ void decode_entry(RansLane<T, TG> &rl, const TableGeom &g, const PostParams &pp, int32_t *prev,
                                             int32_t *v, int32_t *dptr, uint32_t dump, uint64_t e) {
#pragma unroll
  for (int c = 0; c < NCP; ++c) {
    const uint32_t o = rl.template step<CAREFUL, PROBE>();
    const bool compact = TAB == 0 ? g.compact != 0 : TAB == 2;
    const bool zig = MODE == 0 ? g.zig != 0 : MODE != 3;
    v[c] = rl.value(o, compact, zig);
    if (DUMP && (dump & DCB_DUMP_SYMBOLS)) dptr[e * NCP + c] = (int32_t)rl.symbol(o, g);
  }
  const int recon = recon_of<MODE>(pp);
  if (recon == RECON_DELTA_WRAP) {
#pragma unroll
    for (int c = 0; c < NCP; ++c) {
      prev[c] = wrap_original(prev[c], v[c], pp.mn, pp.mx, pp.max_diff);
      v[c] = prev[c];
    }
  } else if (recon == RECON_DELTA_OCT || recon == RECON_DELTA_OCT_CANON) {
    if (NCP == 2) {
      oct_original(pp.box, recon == RECON_DELTA_OCT_CANON, prev[0], prev[NCP - 1], v[0], v[NCP - 1]);
      v[0] = prev[0];
      v[NCP - 1] = prev[NCP - 1];
    }
  }
  if (DUMP && MODE != 3 && (dump & DCB_DUMP_QINTS)) {
#pragma unroll
    for (int c = 0; c < NCP; ++c) dptr[e * NCP + c] = v[c];
  }
}

// SOFTWARE-PIPELINED lean main loop (zig-zag coded corrections, MODE 1..4).  The chain runs ONE SYMBOL AHEAD of the
// post-processing: while the table probe of symbol j is in flight (two dependent LDS, ~60 cycles in which a single
// in-order warp has nothing else to issue), the value map / wrap / dequantisation of symbol j-1 is executed.  ptxas
// left to itself clumps that independent work (profiles/r2_rans_raw_fused_c2_step_cycles.txt); the gate of
// step_lean<.., true> pins the post-processing of symbol j-1 in front of the probe of symbol j+1.
// PROBE: 1 two-region LUT (step_lean), 2 direct slot LUT (step_lean_direct).  COMPACT: the table has a value map.
// One call decodes E entries from entry 4*g on (E a multiple of 4; the LAST group: 4).  Every 4 entries are stored
// and the byte ring is topped up in the body; the wait for those chunks sits in front of the next quad's first byte
// window, not between the last state update and the next renormalisation.  The caller has checked that the bytes of
// the group, and for a middle group those of the next group's first symbol, are there.
template <int NCP, int MODE, bool LAST, int PROBE, bool COMPACT, int E = 4>
__device__ __forceinline__ void lean_sp_group(RansLane<uint16_t, false> &rl, const PostParams &pp, uint8_t *optr, uint32_t g,
                                              int32_t *prev, uint32_t &ca_prev, uint32_t &gate, uint32_t zero) {
  static_assert(E % 4 == 0 && (!LAST || E == 4), "groups of whole quads; the LAST group is one quad");
  constexpr int kQuad = 4 * NCP;  // symbols of 4 entries
  constexpr int kSyms = E * NCP;
#pragma unroll
  for (int qd = 0; qd < E / 4; ++qd) {
    float f[kQuad];
    int32_t v[4][NCP];
#pragma unroll
    for (int t = 1; t <= kQuad; ++t) {
      const int s = qd * kQuad + t;
      uint32_t ca = 0;
      if (!(LAST && s == kSyms)) {
        const int sp = s % kSyms;  // position inside its own group: the windows restart with every group (as run_stream_lean)
        if (sp % 3 == 0) {
          // the quad's first window: every chunk committed before the previous top-up has landed
          if (sp != 0 && sp <= qd * kQuad + 3) cp_async_wait<1>();
          rl.window_open();
        }
        if (PROBE == 2) ca = (sp % 3 == 0) ? rl.template step_lean_direct<true>(gate, zero) : rl.template step_lean_direct<false>(gate, zero);
        else ca = (sp % 3 == 0) ? rl.template step_lean<true, true>(gate, zero) : rl.template step_lean<false, true>(gate, zero);
        if (sp % 3 == 2 || sp == kSyms - 1) rl.window_close();
      }
      const int c = (t - 1) % NCP;
      const int32_t corr = COMPACT ? rl.value_at(ca_prev) : zigzag_dec((ca_prev - rl.cum_addr) >> 1);
      if (MODE == 3 || MODE == 4) prev[c] = corr;  // corrections for oct_chain / the parallelogram kernels
      else prev[c] = wrap_regular(prev[c], corr, pp.mn, pp.mx, pp.max_diff);
      if (MODE == 1) {
        f[t - 1] = pp.dequant(prev[c], c);
        gate = __float_as_uint(f[t - 1]);
      } else {
        v[(t - 1) / NCP][c] = prev[c];
        gate = (uint32_t)corr;  // the value map's load: the integer wrap behind it is three ALU levels
      }
      ca_prev = ca;
    }
    const uint32_t gq = g + (uint32_t)qd;
    if (MODE == 1) {
      float4 *o = reinterpret_cast<float4 *>(reinterpret_cast<float *>(optr) + (uint64_t)gq * kQuad);
#pragma unroll
      for (int k = 0; k < NCP; ++k) o[k] = make_float4(f[4 * k], f[4 * k + 1], f[4 * k + 2], f[4 * k + 3]);
    } else {
      store_group4<NCP>(pp, store_of<MODE>(pp), dsize_of<MODE>(pp), optr, (uint64_t)gq * 4, v);
    }
    rl.template top_up<(4 * NCP * 3 + 15) / 16 + 1>();
  }
}

// Software-pipelined tag loop (see lean_sp_group): the lean chain step -- one byte window per three symbols, two-region
// LUT -- runs one tag ahead; the previous tag's value map sits in the probe's latency shadow (gate).  LAST: the group that
// does not look ahead (the careful tail continues from a clean state).
// PROBE: 1 two-region LUT, 2 direct slot LUT.
template <bool LAST, int PROBE>
__device__ __forceinline__ void tag_sp_group(RansLane<uint16_t, false> &rl, bool compact, uint32_t *t, uint32_t &ca_prev,
                                             uint32_t &gate, uint32_t zero) {
#pragma unroll
  for (int s = 1; s <= 16; ++s) {
    uint32_t ca = 0;
    if (!(LAST && s == 16)) {
      const int sp = s % 16;
      if (sp % 3 == 0) rl.window_open();
      if (PROBE == 2) ca = (sp % 3 == 0) ? rl.template step_lean_direct<true>(gate, zero) : rl.template step_lean_direct<false>(gate, zero);
      else ca = (sp % 3 == 0) ? rl.template step_lean<true, true>(gate, zero) : rl.template step_lean<false, true>(gate, zero);
      if (sp % 3 == 2 || sp == 15) rl.window_close();
    }
    t[s - 1] = rl.value_at_plain(ca_prev, compact) & 0xFFu;  // (byte) cast, SymbolDecoding.cs:41
    gate = t[s - 1];
    ca_prev = ca;
  }
}

template <int PROBE>
__device__ __forceinline__ void run_tags_sp(RansLane<uint16_t, false> &rl, const TableGeom &geom, StreamDesc *dp, uint8_t *aux,
                                            uint32_t zero) {
  const StreamDesc &d = *dp;
  const uint32_t n_entries = d.n_entries;
  const uint32_t ncp = d.ncp;
  const uint64_t avail_bits = (d.buf_end - d.bits_off) * 8ull;
  uint8_t *tags = aux + d.tag_off;
  uint64_t *chunk_bits = reinterpret_cast<uint64_t *>(aux + d.tag_off + (((uint64_t)n_entries + 15ull) & ~15ull));
  const bool compact = geom.compact != 0;
  int status = DCB_OK;
  uint64_t bits = 0;
  uint32_t e = 0;
  // ---- groups of 16 tags (at most 32 bytes), no per-symbol branches; errors are sorted out when the group is left ----
  if (n_entries >= 16u && rl.bytes_left() >= 48u) {
    rl.window_open();
    uint32_t ca_prev = PROBE == 2 ? rl.template step_lean_direct<true>(0u, zero) : rl.template step_lean<true>();
    uint32_t gate = 0;
    for (;;) {
      // a group in the middle looks one tag ahead and leaves enough bytes for the group behind it
      const bool last = !(e + 32u <= n_entries && rl.bytes_left() >= 96u);
      if ((e & (DCB_TAG_CHUNK - 1u)) == 0) chunk_bits[e / DCB_TAG_CHUNK] = bits;
      uint32_t t[16];
      if (last) tag_sp_group<true, PROBE>(rl, compact, t, ca_prev, gate, zero);
      else tag_sp_group<false, PROBE>(rl, compact, t, ca_prev, gate, zero);
      uint32_t tmax = 0, tsum = 0;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        tmax = max(tmax, t[j]);
        tsum += t[j];
      }
      const uint64_t nbits = bits + (uint64_t)tsum * ncp;
      if (tmax > 32u || nbits > avail_bits) {
        // first failing point decides the status, as in the sequential reference loop
        for (int j = 0; j < 16 && status == DCB_OK; ++j) {
          if (t[j] > 32u) status = DCB_ERR_TAG;
          else {
            bits += (uint64_t)t[j] * ncp;
            if (bits > avail_bits) status = DCB_ERR_EOF;
          }
        }
        break;
      }
      uint4 pk;
      pk.x = t[0] | (t[1] << 8) | (t[2] << 16) | (t[3] << 24);
      pk.y = t[4] | (t[5] << 8) | (t[6] << 16) | (t[7] << 24);
      pk.z = t[8] | (t[9] << 8) | (t[10] << 16) | (t[11] << 24);
      pk.w = t[12] | (t[13] << 8) | (t[14] << 16) | (t[15] << 24);
      *reinterpret_cast<uint4 *>(tags + e) = pk;
      bits = nbits;
      e += 16u;
      rl.template top_up<4>();
      cp_async_wait<1>();
      if (last) break;
    }
    rl.prefetch();  // the careful tail reads through the two-word peek
  }
  // ---- careful tail (exact `off > 0` handling, per-point checks) ----
  for (; status == DCB_OK && e < n_entries; ++e) {
    if ((e & (DCB_TAG_CHUNK - 1u)) == 0) chunk_bits[e / DCB_TAG_CHUNK] = bits;
    const uint32_t tag = (uint32_t)rl.value(rl.template step<true, PROBE>(), compact, false) & 0xFFu;
    if (tag > 32u) {
      status = DCB_ERR_TAG;
      break;
    }
    bits += (uint64_t)tag * ncp;
    if (bits > avail_bits) {
      status = DCB_ERR_EOF;
      break;
    }
    tags[e] = (uint8_t)tag;
    rl.top_up<1>();
    cp_async_wait<0>();
  }
  dp->bits_total = bits;
  if (status != DCB_OK) dp->status = status;
}

}  // namespace dcb
