// draco_sharp_b200/csrc/dcb_kernels.cu -- sm_100a kernels of the Draco attribute-decode hot path.
//
// No tensor cores: nothing here is a dense contraction.  The work is serial rANS state chains
// (one chain per compressed attribute stream), integer prediction recurrences and a float
// epilogue.  Parallelism comes from the batch: every lane of a warp owns ONE stream and runs its
// chain; the per-stream probability tables live in that lane's slice of shared memory; the
// compressed bytes are pulled through a register window fed by 16-byte read-only loads issued one
// chunk ahead, so the only latency on the critical path is  smem LUT -> smem cum window -> IMAD ->
// renormalisation.  Everything after the symbol (zig-zag, delta + wrap / octahedron transform,
// dequantisation, store) hangs off the chain and runs in its shadow.
//
// Kernels:
//   rans_raw_fused_kernel   SymbolDecoding.DecodeRawSymbols (Entropy/SymbolDecoding.cs:52-67) + RAnsDecoder.Read
//                           (Entropy/RAnsDecoder.cs:56-99) + zig-zag + PredictionSchemeDeltaDecoder + transform +
//                           dequantise / oct->unit / narrow, in one pass; parallelogram streams emit corrections
//   rans_tag_kernel         the tag half of SymbolDecoding.DecodeTaggedSymbols (SymbolDecoding.cs:30-50)
//   resolve_kernel          continues the container walk behind Tagged bit areas (dcb_walk.h)
//   serial_post_kernel      Tagged bit fields / uncompressed ints / stored corrections -> prediction -> store
//   para_deps_kernel        MeshPredictionSchemeParallelogramDecoder.GetParallelogramEntries (:56-59) for all p
//   para_chain_kernel       MeshPredictionSchemeParallelogramDecoder.ComputeOriginalValues (:29-54)
//   copy_kernel             SequentialAttributeDecoder.DecodeValues (generic attributes, :75-86)
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <stdio.h>
#include <stdlib.h>

#include "dcb_device.cuh"
#include "dcb_internal.h"
#include "dcb_kernels.h"
#include "dcb_walk.h"

using namespace dcb;

namespace {

// ---------------------------------------------------------------------------------------------
// rans_raw_fused: one warp per CTA, `lanes` active lanes, one Raw stream per lane.
// TABLE_GLOBAL: the lane tables live in a global scratch arena instead of shared memory (alphabets
// too large for smem: precision 16..20).
// ---------------------------------------------------------------------------------------------
template <int NCP, typename T, bool DUMP, bool TG, int MODE, int TAB, bool SPLIT>
__device__ __forceinline__ void run_tail(RansLane<T, TG> &rl, const TableGeom &geom, const PostParams &pp, uint8_t *optr,
                                         int32_t *dptr, uint32_t dump, uint32_t n_entries, uint32_t g, int32_t *prev);

// One stream, start to end: main loop over groups of 4 entries, then the careful per-entry tail.
template <int NCP, typename T, bool DUMP, bool TG, int MODE, int TAB, bool SPLIT>
__device__ __forceinline__ void run_stream(RansLane<T, TG> &rl, const TableGeom &geom, const PostParams &pp, uint8_t *optr,
                                           int32_t *dptr, uint32_t dump, uint32_t n_entries, uint32_t g_min) {
  const int store = store_of<MODE>(pp), dsize = dsize_of<MODE>(pp);
  int32_t prev[NCP];
#pragma unroll
  for (int c = 0; c < NCP; ++c) prev[c] = 0;
  // ---- main loop: 4 entries (4 * NCP symbols) per iteration, renormalisation bounds checked once per group ----
  constexpr uint32_t kGroupBytes = 4u * NCP * 3u;
  uint32_t g = 0;
  for (; g < g_min; ++g) {
    if (rl.bytes_left() < kGroupBytes) break;  // per lane: the rest of this stream runs the careful loop
    int32_t v[4][NCP];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      decode_entry<NCP, T, TG, DUMP, MODE, TAB, false, SPLIT>(rl, geom, pp, prev, v[j], dptr, dump, (uint64_t)g * 4 + j);
    store_group4<NCP>(pp, store, dsize, optr, (uint64_t)g * 4, v);
    rl.template top_up<(kGroupBytes + 15) / 16 + 1>();
    cp_async_wait<1>();
  }
  run_tail<NCP, T, DUMP, TG, MODE, TAB, SPLIT>(rl, geom, pp, optr, dptr, dump, n_entries, g, prev);
}

// per-lane tail of a stream: exact `off > 0` handling, one entry at a time
template <int NCP, typename T, bool DUMP, bool TG, int MODE, int TAB, bool SPLIT>
__device__ __forceinline__ void run_tail(RansLane<T, TG> &rl, const TableGeom &geom, const PostParams &pp, uint8_t *optr,
                                         int32_t *dptr, uint32_t dump, uint32_t n_entries, uint32_t g, int32_t *prev) {
  const int store = store_of<MODE>(pp), dsize = dsize_of<MODE>(pp);
  for (uint32_t e = g * 4u; e < n_entries; ++e) {
    int32_t v[NCP];
    decode_entry<NCP, T, TG, DUMP, MODE, TAB, true, SPLIT>(rl, geom, pp, prev, v, dptr, dump, e);
    store_entry<NCP>(pp, store, dsize, optr, e, v);
    rl.template top_up<(3 * NCP + 15) / 16 + 1>();
    cp_async_wait<0>();
  }
}

// LEAN main loop for the hot shape: compact u16 tables in shared memory behind the two-region LUT, delta + wrap on a
// REGULAR stream (see wrap_regular), no debug dumps.  Same group structure as run_stream; per symbol it issues ~1/4
// fewer instructions: the byte supply is one window per three symbols, the renormalisation two predicated funnel
// shifts, the wrap has no clamp.  A warp whose lanes all qualify takes it (vote in the kernel); streams end in the same
// careful tail.
template <int NCP, int MODE>
__device__ __forceinline__ void run_stream_lean(RansLane<uint16_t, false> &rl, const TableGeom &geom, const PostParams &pp,
                                                uint8_t *optr, uint32_t n_entries, uint32_t g_min) {
  const int store = store_of<MODE>(pp), dsize = dsize_of<MODE>(pp);
  int32_t prev[NCP];
  const int32_t p0 = 0 > pp.mx ? pp.mx : (0 < pp.mn ? pp.mn : 0);  // the clamp the first prediction (zero) would get
#pragma unroll
  for (int c = 0; c < NCP; ++c) prev[c] = p0;
  constexpr uint32_t kGroupBytes = 4u * NCP * 3u;
  constexpr int kSyms = 4 * NCP;
  uint32_t g = 0;
  for (; g < g_min; ++g) {
    if (rl.bytes_left() < kGroupBytes) break;
    int32_t v[4][NCP];
#pragma unroll
    for (int s = 0; s < kSyms; ++s) {
      if (s % 3 == 0) rl.window_open();
      const uint32_t ca = (s % 3 == 0) ? rl.template step_lean<true>() : rl.template step_lean<false>();
      if (s % 3 == 2 || s == kSyms - 1) rl.window_close();
      const int32_t corr = rl.value_at(ca);
      const int c = s % NCP;
      prev[c] = wrap_regular(prev[c], corr, pp.mn, pp.mx, pp.max_diff);
      v[s / NCP][c] = prev[c];
    }
    store_group4<NCP>(pp, store, dsize, optr, (uint64_t)g * 4, v);
    rl.template top_up<(kGroupBytes + 15) / 16 + 1>();
    cp_async_wait<1>();
  }
  rl.prefetch();  // the careful tail reads through the two-word peek
  run_tail<NCP, uint16_t, false, false, MODE, 2, true>(rl, geom, pp, optr, nullptr, 0u, n_entries, g, prev);
}

// Software-pipelined lean main loop (lean_sp_group, dcb_device.cuh) around the two-region LUT, E entries per group.
// The bounds are tested once per RUN of groups: a run is as many groups as the lane of `live` with the fewest bytes
// left cannot run out of (step_lean shifts in at most two bytes per symbol), so the groups need no test of their own
// and the loop counter is warp-uniform.  A lane whose own budget is down to zero leaves the run and finishes alone: the
// LAST group, then the careful tail.  `live`: the lanes of the warp that call this.
template <int NCP, int MODE, int E>
__device__ __forceinline__ void run_stream_lean_sp(RansLane<uint16_t, false> &rl, const TableGeom &geom, const PostParams &pp,
                                                   uint8_t *optr, uint32_t n_entries, uint32_t g_min, uint32_t zero,
                                                   uint32_t live) {
  int32_t prev[NCP];
  const int32_t p0 = 0 > pp.mx ? pp.mx : (0 < pp.mn ? pp.mn : 0);  // the clamp the first prediction (zero) would get
#pragma unroll
  for (int c = 0; c < NCP; ++c) prev[c] = p0;
  constexpr uint32_t kQuads = E / 4;
  constexpr uint32_t kMaxGroupBytes = 2u * E * NCP;
  constexpr uint32_t kMargin = 2u * 4u * NCP;  // the symbol in the open window + symbols 1.. of the LAST group
  uint32_t g = 0;  // in groups of 4 entries
  const bool fast = g_min > 0 && rl.bytes_left() >= kMargin;
  uint32_t run = __ballot_sync(live, fast);
  if (fast) {
    // prologue: symbol 0 of group 0 (the window stays open: symbols 1 and 2 follow in the loop)
    rl.window_open();
    uint32_t ca_prev = rl.template step_lean<true>();
    uint32_t gate = 0;
    for (;;) {
      // a middle group leaves at least one group of 4 entries (g_min is the warp's minimum) for the LAST group
      const uint32_t by_bytes = rl.bytes_left() >= kMargin + kMaxGroupBytes ? (rl.bytes_left() - kMargin) / kMaxGroupBytes : 0u;
      const uint32_t mine = min(by_bytes, (g_min - 1u - g) / kQuads);
      run = __ballot_sync(run, mine > 0);
      if (mine == 0) break;
      const uint32_t n = __reduce_min_sync(run, mine);
      for (uint32_t i = 0; i < n; ++i) {
        lean_sp_group<NCP, MODE, false, 1, true, E>(rl, pp, optr, g, prev, ca_prev, gate, zero);
        g += kQuads;
      }
    }
    lean_sp_group<NCP, MODE, true, 1, true>(rl, pp, optr, g, prev, ca_prev, gate, zero);
    ++g;
    cp_async_wait<1>();
  }
  rl.prefetch();  // the careful tail reads through the two-word peek
  run_tail<NCP, uint16_t, false, false, MODE, 2, true>(rl, geom, pp, optr, nullptr, 0u, n_entries, g, prev);
}

template <int NCP, typename T, bool DUMP, bool TABLE_GLOBAL, int MODE, int TAB, int E>
__global__ void __launch_bounds__(32) rans_raw_fused_kernel(const uint8_t *__restrict__ arena, StreamDesc *streams,
                                                            const uint32_t *__restrict__ order, uint32_t n_streams,
                                                            uint32_t lanes, TableGeom geom, uint8_t *__restrict__ out,
                                                            uint8_t *__restrict__ dbg, uint8_t *__restrict__ aux,
                                                            uint8_t *__restrict__ tab_arena, uint32_t dump) {
  extern __shared__ __align__(16) uint8_t smem[];
  const uint32_t lane = threadIdx.x;
  const uint32_t slot = blockIdx.x * lanes + lane;
  const bool have = lane < lanes && slot < n_streams;
  StreamDesc *dp = have ? &streams[order[slot]] : nullptr;
  const uint32_t smem_base = (uint32_t)__cvta_generic_to_shared(smem);
  const SmemLayout lay = smem_layout(smem_base, lanes, geom, TABLE_GLOBAL);

  RansLane<T, TABLE_GLOBAL> rl;
  uint32_t n_entries = 0;
  T *lut = nullptr, *ent = nullptr;
  uint8_t *lutb = nullptr;
  uint32_t *blk = nullptr;
  bool split_ok = true;  // idle lanes do not veto
  bool lean_ok = true;
  if (have) {
    const StreamDesc &d = *dp;
    n_entries = d.n_entries;
    // wide integer attribute (more than 4 components): its n * nc symbols as one-component entries
    if (NCP == 1 && MODE == 0 && d.ncp > 4) n_entries *= d.ncp;
    int status = DCB_OK;
    if (n_entries > 0) {
      uint32_t ent_off;
      if (TABLE_GLOBAL) {
        // per launch slot: [LUT region | entry region] in the global scratch arena
        const uint32_t n_slots = gridDim.x * lanes;
        rl.lut0 = tab_arena;
        rl.ent0 = tab_arena + (size_t)n_slots * geom.lut_bytes;
        rl.lut_base = slot * geom.lut_bytes;
        ent_off = slot * geom.ent_bytes;
        lut = reinterpret_cast<T *>(tab_arena + (size_t)slot * geom.lut_bytes);
        ent = reinterpret_cast<T *>(const_cast<uint8_t *>(rl.ent0) + (size_t)slot * geom.ent_bytes);
      } else {
        rl.lut0 = nullptr;
        rl.ent0 = smem + lay.ent0;
        rl.lut_base = smem_base + lay.lut0 + lane * geom.lut_bytes;
        rl.lutb_addr = smem_base + lay.lutb0 + lane * geom.lutb_bytes;
        rl.blk_addr = smem_base + lay.blk0 + lane * geom.blk_bytes;
        blk = reinterpret_cast<uint32_t *>(smem + lay.blk0 + (size_t)lane * geom.blk_bytes);
        ent_off = lane * geom.ent_bytes;
        rl.cum_addr = smem_base + lay.ent0 + ent_off;
        lut = reinterpret_cast<T *>(smem + lay.lut0 + (size_t)lane * geom.lut_bytes);
        lutb = smem + lay.lutb0 + (size_t)lane * geom.lutb_bytes;
        ent = reinterpret_cast<T *>(smem + lay.ent0 + (size_t)lane * geom.ent_bytes);
      }
      status = rl.build(arena, d, geom, ent, ent_off);
      if (status == DCB_OK) status = rl.init_state(arena, d);
      if (status == DCB_OK) split_ok = rl.split_ok && !(dump & 0x80000000u);
      if (status == DCB_OK) {
        // regular delta + wrap stream (wrap_regular): no correction of the table reaches max_diff, bounds far from int32
        const int64_t md = 1ll + (int64_t)d.xf_b - (int64_t)d.xf_a;
        lean_ok = split_ok && geom.zig != 0 && !(dump & 0x40000000u) &&
                  (MODE == 3 || MODE == 4 ||  // corrections go to the scratch as they are: no wrap to be regular about
                   ((int64_t)rl.max_abs_val < md && d.xf_a >= -(1 << 29) && d.xf_b <= (1 << 29)));
      }
    }
    if (status != DCB_OK) {
      dp->status = status;
      n_entries = 0;
    }
  }
  // the branch-free two-region LUT is used when every stream of the warp can have one
  const bool use_split = __all_sync(0xffffffffu, split_ok);
  const bool use_lean = __all_sync(0xffffffffu, lean_ok);
  // groups of 4 entries every active lane of the warp can run without per-lane bounds checks
  uint32_t g_min = n_entries ? (n_entries >> 2) : 0xFFFFFFFFu;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) g_min = min(g_min, __shfl_xor_sync(0xffffffffu, g_min, o));
  const uint32_t live = __ballot_sync(0xffffffffu, n_entries != 0);
  if (n_entries == 0) return;  // idle lane, empty or failed stream (below, warp-level operations use `live`)
  rl.fill_lut(geom, lut, lutb, blk, ent, use_split);
  rl.init_ring(smem_base + lay.ring0 + lane * DCB_RING_BYTES);

  PostParams pp;
  pp.load(*dp);
  uint8_t *optr = out + dp->out_off;
  int32_t *dptr = DUMP ? reinterpret_cast<int32_t *>(dbg + dp->dbg_off) : nullptr;
  const bool wide_nc = NCP == 1 && MODE == 0 && dp->ncp > 4;
  if (wide_nc) {  // wide_post_kernel reconstructs and dumps the quantized ints
    pp.recon = RECON_NONE;
    dump &= ~(uint32_t)DCB_DUMP_QINTS;
  }
  if (MODE == 3 || MODE == 4 || (MODE == 0 && (pp.recon == RECON_PARA_WRAP || pp.store == STORE_OCT_UNIT || wide_nc))) {
    // int32 scratch: corrections for the parallelogram kernel / for oct_chain_kernel / for wide_post_kernel
    optr = aux + dp->aux_off;
    if (NCP == 2 && pp.store == STORE_OCT_UNIT) {  // normals: the recurrence and its quantized-int dump run in oct_chain_kernel
      pp.recon = RECON_NONE;
      dump &= ~(uint32_t)DCB_DUMP_QINTS;
    }
    pp.store = STORE_NARROW;
    pp.dsize = 4;
  }
  if constexpr (sizeof(T) == 2 && !TABLE_GLOBAL && !DUMP && MODE >= 1 && MODE <= 4 && TAB == 2) {
    // lean main loop: every active lane of the warp decodes a regular delta + wrap stream through the two-region LUT
    if (use_lean) {
#ifndef DCB_NO_LEAN_SP
      run_stream_lean_sp<NCP, MODE, E>(rl, geom, pp, optr, n_entries, g_min, blockIdx.y, live);  // blockIdx.y: an opaque zero
      return;
#endif
      if constexpr (MODE == 1 || MODE == 2) {
        run_stream_lean<NCP, MODE>(rl, geom, pp, optr, n_entries, g_min);
        return;
      }
    }
  }
  if (use_split)
    run_stream<NCP, T, DUMP, TABLE_GLOBAL, MODE, TAB, true>(rl, geom, pp, optr, dptr, dump, n_entries, g_min);
  else
    run_stream<NCP, T, DUMP, TABLE_GLOBAL, MODE, TAB, false>(rl, geom, pp, optr, dptr, dump, n_entries, g_min);
}

// ---------------------------------------------------------------------------------------------
// rans_tag_kernel: the tag stream of a Tagged attribute (32-symbol alphabet, 12-bit precision).
// One stream per lane.  Writes one byte per point (the bit length), the running bit offset at every
// TAG_CHUNK points (for the parallel bit-field extraction) and bits_total; fails the stream on
// tag > 32 (DecoderBuffer.cs:141) or when the bit area would run past the buffer.
// ---------------------------------------------------------------------------------------------
template <bool SPLIT>
__device__ __forceinline__ void run_tags(RansLane<uint16_t, false> &rl, const TableGeom &geom, StreamDesc *dp, uint8_t *aux) {
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
  // ---- groups of 16 tags, no per-symbol branches; errors are sorted out when the group is left ----
  for (; e + 16 <= n_entries; e += 16) {
    if (rl.bytes_left() < 48u) break;  // renormalisation may run out of bytes: careful loop below
    if ((e & (DCB_TAG_CHUNK - 1u)) == 0) chunk_bits[e / DCB_TAG_CHUNK] = bits;
    uint32_t t[16];
#pragma unroll
    for (int j = 0; j < 16; ++j)
      t[j] = (uint32_t)rl.value(rl.template step<false, SPLIT>(), compact, false) & 0xFFu;  // (byte) cast, SymbolDecoding.cs:41
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
    rl.template top_up<4>();
    cp_async_wait<1>();
  }
  // ---- careful tail (exact `off > 0` handling, per-point checks) ----
  for (; status == DCB_OK && e < n_entries; ++e) {
    if ((e & (DCB_TAG_CHUNK - 1u)) == 0) chunk_bits[e / DCB_TAG_CHUNK] = bits;
    const uint32_t tag = (uint32_t)rl.value(rl.template step<true, SPLIT>(), compact, false) & 0xFFu;
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

__global__ void __launch_bounds__(32) rans_tag_kernel(const uint8_t *__restrict__ arena, StreamDesc *streams,
                                                      const uint32_t *__restrict__ order, uint32_t n_streams,
                                                      uint32_t lanes, TableGeom geom, uint8_t *__restrict__ aux) {
  extern __shared__ __align__(16) uint8_t smem[];
  typedef uint16_t T;
  const uint32_t lane = threadIdx.x;
  const uint32_t slot = blockIdx.x * lanes + lane;
  const bool have = lane < lanes && slot < n_streams;
  StreamDesc *dp = have ? &streams[order[slot]] : nullptr;
  const uint32_t smem_base = (uint32_t)__cvta_generic_to_shared(smem);
  const SmemLayout lay = smem_layout(smem_base, lanes, geom, false);
  RansLane<T, false> rl;
  T *ent = reinterpret_cast<T *>(smem + lay.ent0 + (size_t)lane * geom.ent_bytes);
  bool alive = false, split_ok = true;
  if (have) {
    rl.lut0 = nullptr;
    rl.ent0 = smem + lay.ent0;
    rl.lut_base = smem_base + lay.lut0 + lane * geom.lut_bytes;
    rl.lutb_addr = smem_base + lay.lutb0 + lane * geom.lutb_bytes;
    rl.blk_addr = smem_base + lay.blk0 + lane * geom.blk_bytes;
    rl.cum_addr = smem_base + lay.ent0 + lane * geom.ent_bytes;
    int status = rl.build(arena, *dp, geom, ent, lane * geom.ent_bytes);
    if (status == DCB_OK) status = rl.init_state(arena, *dp);
    if (status != DCB_OK) {
      dp->status = status;
      dp->bits_total = 0;
    } else {
      alive = true;
      split_ok = rl.split_ok;
    }
  }
  const bool use_split = __all_sync(0xffffffffu, split_ok);
  if (!alive) return;
  rl.fill_lut(geom, reinterpret_cast<T *>(smem + lay.lut0 + (size_t)lane * geom.lut_bytes),
              smem + lay.lutb0 + (size_t)lane * geom.lutb_bytes,
              reinterpret_cast<uint32_t *>(smem + lay.blk0 + (size_t)lane * geom.blk_bytes), ent, use_split);
  rl.init_ring(smem_base + lay.ring0 + lane * DCB_RING_BYTES);
#ifndef DCB_NO_LEAN_SP
  if (use_split) run_tags_sp<1>(rl, geom, dp, aux, blockIdx.y);  // blockIdx.y: an opaque zero
  else
#endif
  if (use_split) run_tags<true>(rl, geom, dp, aux);
  else run_tags<false>(rl, geom, dp, aux);
}

// ---------------------------------------------------------------------------------------------
// resolve_kernel: one thread per buffer whose walk stopped at a Tagged bit area.
// ---------------------------------------------------------------------------------------------
__global__ void resolve_kernel(const uint8_t *__restrict__ arena, BufWalk *walks, const uint32_t *__restrict__ list,
                               uint32_t n, StreamDesc *streams) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  BufWalk w = walks[list[i]];
  walk_continue(arena, w, streams);
  walks[list[i]] = w;
  // a walk that failed behind the bit area fails every stream of its buffer: the host may have launched their kernels
  // without waiting for this verdict (a Tagged attribute that closes its buffer needs no round trip)
  if (w.status != DCB_OK)
    for (int k = 0; k < w.stream_count; ++k)
      if (streams[w.stream_first + k].status == DCB_OK) streams[w.stream_first + k].status = w.status;
}

// ---------------------------------------------------------------------------------------------
// serial_post_kernel: one stream per lane; sources that need no rANS chain.
//   Tagged        tags (u8 per point, from rans_tag_kernel) + LSB-first bit fields (DecoderBuffer.cs:138-154, B-4)
//   Uncompressed  raw_num_bytes little-endian bytes per value (SequentialIntegerAttributeDecoder.cs:68-84, B-6)
//   Empty         n_entries * ncp == 0
// followed by zig-zag, the serial prediction recurrence and the store.  This is the path for
// octahedron transforms and irregular wrap streams behind a Tagged source, and the general fallback.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t read_bits_lsb(const uint8_t *p, uint64_t bitpos, uint32_t count) {
  if (count == 0) return 0;
  const uint64_t byte = bitpos >> 3;
  const uint32_t sh = (uint32_t)(bitpos & 7u);
  uint64_t w = 0;
  const uint32_t need = (sh + count + 7u) >> 3;  // <= 5
  for (uint32_t k = 0; k < need; ++k) w |= (uint64_t)p[byte + k] << (8u * k);
  w >>= sh;
  return count == 32 ? (uint32_t)w : ((uint32_t)w & ((1u << count) - 1u));
}

template <int NCP, bool DUMP>
__global__ void __launch_bounds__(32) serial_post_kernel(const uint8_t *__restrict__ arena, StreamDesc *streams,
                                                         const uint32_t *__restrict__ order, uint32_t n_streams,
                                                         uint8_t *__restrict__ out, uint8_t *__restrict__ dbg,
                                                         uint8_t *__restrict__ aux, uint32_t dump,
                                                         uint32_t only_irregular) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_streams) return;
  StreamDesc &d = streams[order[slot]];
  if (d.status != DCB_OK) return;
  if (only_irregular && !d.irregular) return;  // the point-parallel kernels decoded it
  const uint32_t n_entries = d.n_entries;
  PostParams pp;
  pp.load(d);
  uint8_t *optr = out + d.out_off;
  int32_t *dptr = DUMP ? reinterpret_cast<int32_t *>(dbg + d.dbg_off) : nullptr;
  if (pp.recon == RECON_PARA_WRAP || pp.store == STORE_OCT_UNIT) {
    optr = aux + d.aux_off;
    pp.store = STORE_NARROW;
    pp.dsize = 4;
  }
  const uint8_t scheme = d.scheme;
  const uint8_t *tags = aux + d.tag_off;
  const uint8_t *bits = arena + d.bits_off;
  const uint8_t *raw = arena + d.raw_off;
  const uint32_t nb = d.raw_num_bytes;
  uint64_t bitpos = 0;
  int32_t prev[NCP];
#pragma unroll
  for (int c = 0; c < NCP; ++c) prev[c] = 0;
  for (uint32_t e = 0; e < n_entries; ++e) {
    int32_t v[NCP];
    uint32_t tag = 0;
    if (scheme == SCHEME_TAGGED) tag = tags[e];
#pragma unroll
    for (int c = 0; c < NCP; ++c) {
      uint32_t sym = 0;
      if (scheme == SCHEME_TAGGED) {
        sym = read_bits_lsb(bits, bitpos, tag);
        bitpos += tag;
      } else {
        const uint8_t *q = raw + ((uint64_t)e * NCP + c) * nb;
        for (uint32_t k = 0; k < nb; ++k) sym |= (uint32_t)q[k] << (8u * k);
      }
      if (DUMP && (dump & DCB_DUMP_SYMBOLS)) dptr[(size_t)e * NCP + c] = (int32_t)sym;
      v[c] = pp.zig ? zigzag_dec(sym) : (int32_t)sym;
    }
    if (pp.recon == RECON_DELTA_WRAP) {
#pragma unroll
      for (int c = 0; c < NCP; ++c) {
        prev[c] = wrap_original(prev[c], v[c], pp.mn, pp.mx, pp.max_diff);
        v[c] = prev[c];
      }
    } else if (pp.recon == RECON_DELTA_OCT || pp.recon == RECON_DELTA_OCT_CANON) {
      if (NCP == 2) {
        oct_original(pp.box, pp.recon == RECON_DELTA_OCT_CANON, prev[0], prev[NCP - 1], v[0], v[NCP - 1]);
        v[0] = prev[0];
        v[NCP - 1] = prev[NCP - 1];
      }
    }
    if (DUMP && (dump & DCB_DUMP_QINTS) && pp.recon != RECON_PARA_WRAP) {
#pragma unroll
      for (int c = 0; c < NCP; ++c) dptr[(size_t)e * NCP + c] = v[c];
    }
    store_entry<NCP>(pp, pp.store, pp.dsize, optr, e, v);
  }
}

// wide_post_kernel: integer attributes with MORE THAN 4 components (the reference loops over any nc:
// SequentialIntegerAttributeDecoder.cs:53-101 for the values, :142-160 for the narrowing store).  One stream per lane,
// run-time component count, running values of the delta decoder in local memory.  Sources: the zig-zag decoded symbols
// a Raw stream left in the scratch (fused kernel, one-component instantiation), tags + bit fields, or uncompressed
// values.  Rare shapes (joint indices / weights beyond 4, custom vectors): correctness, not speed.
template <bool DUMP>
__global__ void __launch_bounds__(32) wide_post_kernel(const uint8_t *__restrict__ arena, StreamDesc *streams,
                                                       const uint32_t *__restrict__ order, uint32_t n_streams,
                                                       uint8_t *__restrict__ out, uint8_t *__restrict__ dbg,
                                                       uint8_t *__restrict__ aux, uint32_t dump) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_streams) return;
  StreamDesc &d = streams[order[slot]];
  if (d.status != DCB_OK) return;
  const uint32_t n_entries = d.n_entries, nc = d.ncp;
  PostParams pp;
  pp.load(d);
  uint8_t *optr = out + d.out_off;
  int32_t *dptr = DUMP ? reinterpret_cast<int32_t *>(dbg + d.dbg_off) : nullptr;
  const uint8_t scheme = d.scheme;
  const int32_t *corr = reinterpret_cast<const int32_t *>(aux + d.aux_off);
  const uint8_t *tags = aux + d.tag_off;
  const uint8_t *bits = arena + d.bits_off;
  const uint8_t *raw = arena + d.raw_off;
  const uint32_t nb = d.raw_num_bytes;
  const int dsize = dcb_dtype_len(d.data_type);
  uint64_t bitpos = 0;
  int32_t prev[256];
  for (uint32_t c = 0; c < nc; ++c) prev[c] = 0;
  for (uint32_t e = 0; e < n_entries; ++e) {
    uint32_t tag = 0;
    if (scheme == SCHEME_TAGGED) tag = tags[e];
    for (uint32_t c = 0; c < nc; ++c) {
      const uint64_t i = (uint64_t)e * nc + c;
      int32_t v;
      if (scheme == SCHEME_RAW) {
        v = corr[i];  // value map of the fused kernel: zig-zag decoded already (or the plain symbol when !zig)
      } else {
        uint32_t sym = 0;
        if (scheme == SCHEME_TAGGED) {
          sym = read_bits_lsb(bits, bitpos, tag);
          bitpos += tag;
        } else if (scheme == SCHEME_UNCOMPRESSED) {
          const uint8_t *q = raw + i * nb;
          for (uint32_t k = 0; k < nb; ++k) sym |= (uint32_t)q[k] << (8u * k);
        }
        if (DUMP && (dump & DCB_DUMP_SYMBOLS)) dptr[i] = (int32_t)sym;
        v = pp.zig ? zigzag_dec(sym) : (int32_t)sym;
      }
      if (pp.recon == RECON_DELTA_WRAP) {
        prev[c] = wrap_original(prev[c], v, pp.mn, pp.mx, pp.max_diff);
        v = prev[c];
      }
      if (DUMP && (dump & DCB_DUMP_QINTS)) dptr[i] = v;
      if (dsize == 1) optr[i] = (uint8_t)v;
      else if (dsize == 2) reinterpret_cast<uint16_t *>(optr)[i] = (uint16_t)v;
      else reinterpret_cast<int32_t *>(optr)[i] = v;
    }
  }
}

// par_post2_kernel (the point-parallel path behind Tagged / uncompressed sources) lives in dcb_par_post.cu.

// ---------------------------------------------------------------------------------------------
// parallelogram prediction
// ---------------------------------------------------------------------------------------------
// deps[p] = (opp, next, prev) entry ids of the parallelogram of entry p, or (-1,*,*) when the
// predictor falls back to entry p-1.  Depends on the connectivity maps only: fully parallel.
__global__ void para_deps_kernel(StreamDesc *streams, const uint32_t *__restrict__ order, uint32_t n_streams,
                                 const uint8_t *__restrict__ maps, uint8_t *__restrict__ aux) {
  for (uint32_t si = blockIdx.y; si < n_streams; si += gridDim.y) {
  StreamDesc &d = streams[order[si]];
  if (d.status != DCB_OK) continue;
  const uint32_t n = d.n_entries;
  const uint32_t *opp = reinterpret_cast<const uint32_t *>(maps + d.map_off[0]);
  const uint32_t *c2v = reinterpret_cast<const uint32_t *>(maps + d.map_off[1]);
  const uint32_t *d2c = reinterpret_cast<const uint32_t *>(maps + d.map_off[2]);
  const int32_t *v2d = reinterpret_cast<const int32_t *>(maps + d.map_off[3]);
  const uint32_t n_corners = d.n_corners, n_vertices = d.n_vertices;
  // deps live behind the corrections in the stream's scratch: int32[n * ncp] | qints int32[n * ncp] | int32[3 n]
  int32_t *deps = reinterpret_cast<int32_t *>(aux + d.aux_off) + 2ull * n * d.ncp;
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
    int32_t e_o = -1, e_n = -1, e_p = -1;
    if (p > 0) {
      const uint32_t corner = d2c[p];
      if (corner != 0xFFFFFFFFu && corner < n_corners) {
        const uint32_t oc = opp[corner];  // MeshPredictionSchemeParallelogramDecoder.cs:66
        if (oc != 0xFFFFFFFFu) {
          if (oc >= n_corners) {
            d.status = DCB_ERR_MAPS;
          } else {
            const uint32_t nx = (oc % 3u == 2u) ? oc - 2u : oc + 1u;  // CornerTable.Next
            const uint32_t pv = (oc % 3u == 0u) ? oc + 2u : oc - 1u;  // CornerTable.Previous
            const uint32_t v_o = c2v[oc], v_n = c2v[nx], v_p = c2v[pv];
            if (v_o >= n_vertices || v_n >= n_vertices || v_p >= n_vertices) {
              d.status = DCB_ERR_MAPS;
            } else {
              const int32_t a = v2d[v_o], b = v2d[v_n], c = v2d[v_p];
              if (a < (int32_t)p && b < (int32_t)p && c < (int32_t)p) {  // :75
                if (a < 0 || b < 0 || c < 0) d.status = DCB_ERR_MAPS;
                else { e_o = a; e_n = b; e_p = c; }
              }
            }
          }
        }
      }
    }
    deps[3ull * p] = e_o;
    deps[3ull * p + 1] = e_n;
    deps[3ull * p + 2] = e_p;
  }
  }
}

// The recurrence itself.  Its dependency graph is a chain in practice (a depth-first traversal predicts almost every
// entry from the one decoded just before it: dependency depth 1,529 of 1,775 entries on the reference's sample mesh), so
// the "wavefront" is one entry wide inside a stream and the parallelism is across streams: ONE CTA OF TWO WARPS PER
// STREAM, in lock step over blocks of 64 entries.
//   chain warp   lanes 0..NCP-1 walk the chain, one component each (components never mix).  Per entry and component the
//                helper has prepared a record {address of operand opp, next, prev, correction} and a coefficient k:
//                pred = v(next) + v(prev) - v(opp) + k * value(p-1).  An operand that IS entry p-1 points at a zero
//                word and counts in k, so the value of entry p-1 never leaves its register; an entry predicted from
//                p-1 alone (no parallelogram) has three zero operands and k = 1.  No branch, no select, ~20
//                instructions per entry; records of entry p+2 and operands of p+1 are in flight while p is computed.
//   helper warp  runs around the chain: stores the finished block b-1 (quantized ints for later gathers, dequantised
//                output, coalesced), cp.asyncs the dependencies / corrections of block b+2, GATHERS the operands of
//                block b+1 that were decoded before block b started (anything older than the 128-entry history ring)
//                from the quantized-int scratch, and writes block b+1's records.
constexpr uint32_t kParaBlock = 64;    // entries per block
constexpr uint32_t kParaHist = 128;    // history ring: the block being decoded and the one before it

__device__ __forceinline__ void cp_async4(uint32_t smem_addr, const void *gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(smem_addr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ int32_t lds32(uint32_t smem_addr) {
  int32_t v;
  asm volatile("ld.shared.b32 %0, [%1];\n" : "=r"(v) : "r"(smem_addr) : "memory");
  return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t smem_addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_addr) : "memory");
  return v;
}

template <int NCP, bool DUMP>
__global__ void __launch_bounds__(64) para_chain_kernel(StreamDesc *streams, const uint32_t *__restrict__ order,
                                                        uint32_t n_streams, uint8_t *__restrict__ out,
                                                        uint8_t *__restrict__ dbg, uint8_t *__restrict__ aux,
                                                        uint32_t dump) {
  __shared__ int32_t s_dep[3][kParaBlock * 3];           // (opp, next, prev) entry ids; -1 = predict from entry p-1
  __shared__ int32_t s_cor[3][kParaBlock * NCP];         // corrections
  __shared__ int32_t s_far[2][kParaBlock * 3 * NCP];     // gathered operands older than the history ring
  __shared__ __align__(16) uint4 s_rec[2][kParaBlock * NCP];  // {addr opp, addr next, addr prev, correction}
  __shared__ int32_t s_k[2][kParaBlock];                 // coefficient of value(p-1)
  __shared__ int32_t s_hist[kParaHist * NCP];
  __shared__ int32_t s_zero;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const uint32_t a_hist0 = (uint32_t)__cvta_generic_to_shared(s_hist);
  const uint32_t a_zero = (uint32_t)__cvta_generic_to_shared(&s_zero);
  for (uint32_t si = blockIdx.x; si < n_streams; si += gridDim.x) {
    StreamDesc &d = streams[order[si]];
    if (d.status != DCB_OK) continue;   // uniform over the CTA
    const uint32_t n = d.n_entries;
    if (n == 0) continue;
    PostParams pp;
    pp.load(d);
    uint8_t *optr = out + d.out_off;
    int32_t *dptr = DUMP ? reinterpret_cast<int32_t *>(dbg + d.dbg_off) : nullptr;
    const int32_t *corr = reinterpret_cast<const int32_t *>(aux + d.aux_off);
    int32_t *qints = reinterpret_cast<int32_t *>(aux + d.aux_off) + (uint64_t)n * NCP;
    const int32_t *deps = qints + (uint64_t)n * NCP;
    const uint32_t n_blocks = (n + kParaBlock - 1) / kParaBlock;
    // ---- helper warp's pieces ----
    auto stage = [&](uint32_t blk) {  // dependencies + corrections of block blk -> shared memory
      if (blk >= n_blocks) return;
      const uint32_t e0 = blk * kParaBlock, cnt = min(kParaBlock, n - e0), b = blk % 3u;
      for (uint32_t i = lane; i < cnt * 3; i += 32)
        cp_async4((uint32_t)__cvta_generic_to_shared(&s_dep[b][i]), deps + 3ull * e0 + i);
      for (uint32_t i = lane; i < cnt * NCP; i += 32)
        cp_async4((uint32_t)__cvta_generic_to_shared(&s_cor[b][i]), corr + (uint64_t)e0 * NCP + i);
    };
    auto gather = [&](uint32_t blk) {  // operands of block blk decoded before block blk-1 started
      if (blk >= n_blocks || blk < 2) return;
      const uint32_t e0 = blk * kParaBlock, cnt = min(kParaBlock, n - e0), b = blk % 3u, limit = e0 - kParaBlock;
      for (uint32_t i = lane; i < cnt * 3; i += 32) {
        const int32_t e = s_dep[b][i];
        if (s_dep[b][i - i % 3u] >= 0 && (uint32_t)e < limit) {
#pragma unroll
          for (int c = 0; c < NCP; ++c)
            cp_async4((uint32_t)__cvta_generic_to_shared(&s_far[blk & 1u][i * NCP + c]), qints + (uint64_t)(uint32_t)e * NCP + c);
        }
      }
    };
    auto records = [&](uint32_t blk) {  // block blk's operand addresses and coefficients (needs its dependencies)
      if (blk >= n_blocks) return;
      const uint32_t e0 = blk * kParaBlock, cnt = min(kParaBlock, n - e0), b = blk % 3u;
      const uint32_t limit = e0 >= kParaBlock ? e0 - kParaBlock : 0u;
      const uint32_t a_far = (uint32_t)__cvta_generic_to_shared(s_far[blk & 1u]);
      for (uint32_t i = lane; i < cnt * NCP; i += 32) {
        const uint32_t j = i / NCP, c = i - j * NCP, p = e0 + j;
        const int32_t e_o = s_dep[b][3 * j], e_n = s_dep[b][3 * j + 1], e_p = s_dep[b][3 * j + 2];
        const bool para = e_o >= 0;
        int32_t k = para ? 0 : 1;
        auto addr = [&](int32_t e, uint32_t which, int32_t sign) -> uint32_t {
          if (!para) return a_zero;
          if ((uint32_t)e + 1u == p) { k += sign; return a_zero; }
          if ((uint32_t)e < limit) return a_far + ((3u * j + which) * NCP + c) * 4u;
          return a_hist0 + (((uint32_t)e & (kParaHist - 1u)) * NCP + c) * 4u;
        };
        uint4 r;
        r.x = addr(e_o, 0, -1);
        r.y = addr(e_n, 1, 1);
        r.z = addr(e_p, 2, 1);
        r.w = (uint32_t)s_cor[b][i];
        s_rec[blk & 1u][i] = r;
        if (c == 0) s_k[blk & 1u][j] = k;
      }
    };
    auto output = [&](uint32_t blk) {  // finished block -> quantized-int scratch (later gathers read it), dump, typed output
      const uint32_t e0 = blk * kParaBlock, cnt = min(kParaBlock, n - e0);
      for (uint32_t j = lane; j < cnt; j += 32) {
        const uint32_t p = e0 + j;
        int32_t v[NCP];
#pragma unroll
        for (int c = 0; c < NCP; ++c) v[c] = s_hist[(p & (kParaHist - 1u)) * NCP + c];
#pragma unroll
        for (int c = 0; c < NCP; ++c) qints[(uint64_t)p * NCP + c] = v[c];
        if (DUMP && (dump & DCB_DUMP_QINTS)) {
#pragma unroll
          for (int c = 0; c < NCP; ++c) dptr[(size_t)p * NCP + c] = v[c];
        }
        store_entry<NCP>(pp, pp.store, pp.dsize, optr, p, v);
      }
    };
    __syncthreads();  // the previous stream's last block has left shared memory
    if (threadIdx.x == 0) s_zero = 0;
    if (warp == 1) {
      stage(0);
      stage(1);
      cp_async_commit();
      cp_async_wait<0>();
      __syncwarp();
      records(0);
    }
    __syncthreads();
    int32_t prev = 0;  // chain lanes: value of entry p-1, component `lane`
    for (uint32_t blk = 0; blk < n_blocks; ++blk) {
      if (warp == 0) {
        if (lane < NCP) {
          const uint32_t e0 = blk * kParaBlock, cnt = min(kParaBlock, n - e0);
          const uint32_t a_rec = (uint32_t)__cvta_generic_to_shared(s_rec[blk & 1u]) + 16u * lane;
          const uint32_t a_k = (uint32_t)__cvta_generic_to_shared(s_k[blk & 1u]);
          const uint32_t a_st = a_hist0 + ((e0 & (kParaHist - 1u)) * NCP + lane) * 4u;  // a block never wraps the ring
          // two-deep software pipeline: record of entry j+2 and operands of entry j+1 in flight while j is computed
          uint4 r1 = lds128(a_rec);
          int32_t k1 = lds32(a_k);
          int32_t vo = lds32(r1.x), va = lds32(r1.y), vb = lds32(r1.z), co = (int32_t)r1.w, kk = k1;
          const uint32_t j1 = cnt > 1 ? 1u : 0u;
          r1 = lds128(a_rec + j1 * (16u * NCP));
          k1 = lds32(a_k + 4u * j1);
          for (uint32_t j = 0; j < cnt; ++j) {
            const uint32_t j2 = j + 2 < cnt ? j + 2 : j;  // harmless re-read at the end of the block
            const uint4 r2 = lds128(a_rec + j2 * (16u * NCP));
            const int32_t k2 = lds32(a_k + 4u * j2);
            // operands of entry j+1: history up to entry j-1 is in shared memory, entry j itself rides in k
            const int32_t nvo = lds32(r1.x), nva = lds32(r1.y), nvb = lds32(r1.z);
            const int32_t sum = (int32_t)((uint32_t)va + (uint32_t)vb - (uint32_t)vo);
            const int32_t pred = (int32_t)((uint32_t)sum + (uint32_t)kk * (uint32_t)prev);  // :84 / :36,:49-50
            prev = wrap_original(pred, co, pp.mn, pp.mx, pp.max_diff);
            asm volatile("st.shared.b32 [%0], %1;\n" ::"r"(a_st + j * (4u * NCP)), "r"(prev) : "memory");
            vo = nvo; va = nva; vb = nvb; co = (int32_t)r1.w; kk = k1;
            r1 = r2; k1 = k2;
          }
        }
      } else {
        if (blk > 0) output(blk - 1);
        __syncwarp();
        stage(blk + 2);
        gather(blk + 1);   // the scratch now holds every entry before block blk
        cp_async_commit();
        records(blk + 1);
        cp_async_wait<0>();
        __syncwarp();
      }
      __syncthreads();
    }
    if (warp == 1) output(n_blocks - 1);
  }
}

// PredictionSchemeDeltaDecoder over PredictionSchemeNormalOctahedron(Canonicalized)DecodingTransform
// (ComputeOriginalValue, :34-78): orig[i] = f(orig[i-1], corr[i]) on the int32 pairs the Raw rANS kernel (MODE 3) left
// in the stream's scratch, in place.  One stream per lane, no shared memory: the kernel shares the SMs with whatever
// rANS kernels of the batch are running.  Four entries per iteration, the next four prefetched.
template <bool DUMP>
__global__ void __launch_bounds__(32) oct_chain_kernel(StreamDesc *streams, const uint32_t *__restrict__ order,
                                                       uint32_t n_streams, uint8_t *__restrict__ aux,
                                                       uint8_t *__restrict__ dbg, uint32_t dump) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_streams) return;
  const StreamDesc &d = streams[order[slot]];
  if (d.status != DCB_OK) return;
  if (d.recon != RECON_DELTA_OCT && d.recon != RECON_DELTA_OCT_CANON) return;  // geometric normals: geo_normal_kernel
  const uint32_t n = d.n_entries;
  PostParams pp;
  pp.load(d);
  const bool canonical = d.recon == RECON_DELTA_OCT_CANON;
  int4 *st = reinterpret_cast<int4 *>(aux + d.aux_off);  // two (s, t) pairs per int4; scratch offsets are 16-byte aligned
  int32_t *dptr = DUMP ? reinterpret_cast<int32_t *>(dbg + d.dbg_off) : nullptr;
  int32_t p0 = 0, p1 = 0;
  const uint32_t n4 = n / 4;
  int4 a = make_int4(0, 0, 0, 0), b = a;
  if (n4) { a = st[0]; b = st[1]; }
  for (uint32_t g = 0; g < n4; ++g) {
    int4 na = a, nb = b;
    if (g + 1 < n4) { na = st[2 * g + 2]; nb = st[2 * g + 3]; }
    oct_original(pp.box, canonical, p0, p1, a.x, a.y);
    a.x = p0; a.y = p1;
    oct_original(pp.box, canonical, p0, p1, a.z, a.w);
    a.z = p0; a.w = p1;
    oct_original(pp.box, canonical, p0, p1, b.x, b.y);
    b.x = p0; b.y = p1;
    oct_original(pp.box, canonical, p0, p1, b.z, b.w);
    b.z = p0; b.w = p1;
    st[2 * g] = a;
    st[2 * g + 1] = b;
    if (DUMP && (dump & DCB_DUMP_QINTS)) {
      reinterpret_cast<int4 *>(dptr)[2 * g] = a;
      reinterpret_cast<int4 *>(dptr)[2 * g + 1] = b;
    }
    a = na;
    b = nb;
  }
  int2 *s2 = reinterpret_cast<int2 *>(aux + d.aux_off);
  for (uint32_t e = n4 * 4; e < n; ++e) {
    int2 c = s2[e];
    oct_original(pp.box, canonical, p0, p1, c.x, c.y);
    c.x = p0; c.y = p1;
    s2[e] = c;
    if (DUMP && (dump & DCB_DUMP_QINTS)) reinterpret_cast<int2 *>(dptr)[e] = c;
  }
}

// AttributeOctahedronTransform.InverseTransformAttribute (:82-102): quantized octahedral (s, t) -> unit vector,
// one thread per entry, reading the int32 pairs the serial kernels left in scratch
__global__ void oct_unit_kernel(StreamDesc *streams, const uint32_t *__restrict__ order, uint32_t n_streams,
                                uint8_t *__restrict__ out, const uint8_t *__restrict__ aux) {
  for (uint32_t si = blockIdx.y; si < n_streams; si += gridDim.y) {
    const StreamDesc &d = streams[order[si]];
    if (d.status != DCB_OK) continue;
    if (d.recon == RECON_GEO_OCT || d.recon == RECON_GEO_OCT_CANON) continue;  // geo_normal_kernel stores the unit vectors itself
    const int32_t max_value = (int32_t)((1u << d.q_bits) - 2u);
    const float scale = __fdiv_rn(2.0f, __int2float_rn(max_value));  // OctahedronToolBox.cs:19
    const int2 *st = reinterpret_cast<const int2 *>(aux + d.aux_off);
    float *o = reinterpret_cast<float *>(out + d.out_off);
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < d.n_entries; e += gridDim.x * blockDim.x) {
      const int2 q = st[e];
      float x, y, z;
      oct_to_unit(q.x, q.y, scale, x, y, z);
      o[3ull * e] = x;
      o[3ull * e + 1] = y;
      o[3ull * e + 2] = z;
    }
  }
}

// generic attributes: n * byte_stride raw bytes
__global__ void copy_kernel(const uint8_t *__restrict__ arena, StreamDesc *streams, const uint32_t *__restrict__ order,
                            uint32_t n_streams, uint8_t *__restrict__ out) {
  for (uint32_t si = blockIdx.y; si < n_streams; si += gridDim.y) {
    const StreamDesc &d = streams[order[si]];
    if (d.status != DCB_OK) continue;
    const uint8_t *src = arena + d.raw_off;
    uint8_t *dst = out + d.out_off;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < d.out_bytes; i += (uint64_t)gridDim.x * blockDim.x)
      dst[i] = src[i];
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------
static TableGeom geom_of(const RansLaunch &p) {
  TableGeom g{};
  g.lut_bytes = p.lut_bytes;
  g.lutb_bytes = p.lutb_bytes;
  g.blk_bytes = p.lutb_bytes ? (((1u << p.prec_bits) >> 7) << 2) : 0u;
  if (g.blk_bytes && g.blk_bytes < 16u) g.blk_bytes = 16u;
  g.ent_bytes = p.ent_bytes;
  g.cap_entries = p.cap_entries;
  g.cap_exc = p.cap_exc;
  g.lut_shift = p.lut_shift;
  g.compact = p.compact;
  g.zig = p.zig;
  return g;
}

uint32_t dcb_rans_smem_bytes(const RansLaunch &p, bool table_global) {
  // worst-case alignment slack + LUTs + rings + entries (see smem_layout)
  uint32_t b = DCB_RING_BYTES + p.lanes_per_warp * DCB_RING_BYTES;
  if (!table_global && p.direct) return b + 32u + p.lanes_per_warp * (p.lut_bytes + p.ent_bytes);  // direct slot LUT: 16-byte alignment only
  if (!table_global) {
    const uint32_t blk = p.lutb_bytes ? std::max(16u, ((1u << p.prec_bits) >> 7) << 2) : 0u;
    b += p.lut_bytes + blk + 16u + p.lanes_per_warp * (p.lut_bytes + p.lutb_bytes + blk + p.ent_bytes);
  }
  return b;
}

// DCB_NO_SPLIT=1 forces the uniform-LUT probe (tests of the fallback path): bit 31 of the kernel's `dump` word;
// DCB_NO_LEAN=1 keeps regular streams on the general main loop (A/B measurements, tests): bit 30
static uint32_t no_split_bit() {
  static const uint32_t bit = (getenv("DCB_NO_SPLIT") ? 0x80000000u : 0u) | (getenv("DCB_NO_LEAN") ? 0x40000000u : 0u);
  return bit;
}

// entries per group of the software-pipelined lean loop (run_stream_lean_sp); DCB_LEAN_GROUP=4|8|16 picks another
// instance (A/B measurements, tests), any other value keeps the default.  8 measures best on configs[1] (DESIGN 3.1,
// profiles/lean_group_b200.jsonl): 4 pays the group boundary twice as often, 16's unrolled body (~2,900 SASS
// instructions, 46 KB) runs 30 % slower than 8's.
constexpr int kLeanGroup = 8;
static int lean_group() {
  static const int e = [] {
    const char *v = getenv("DCB_LEAN_GROUP");
    const int x = v ? atoi(v) : 0;
    return (x == 4 || x == 8 || x == 16) ? x : kLeanGroup;
  }();
  return e;
}

template <int NCP, typename T, bool DUMP, bool TG, int MODE, int TAB = 0, int E = 4>
static cudaError_t launch_raw_t(const RansLaunch &p, const DevArenas &a, cudaStream_t st) {
  auto k = rans_raw_fused_kernel<NCP, T, DUMP, TG, MODE, TAB, E>;
  const uint32_t smem_bytes = dcb_rans_smem_bytes(p, TG);
  if (smem_bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (e != cudaSuccess) return e;
  }
  // the whole SM as shared memory, whatever this launch needs: CTAs of other launches (pipeline slices, side-stream
  // groups) can only move in next to ours when the carve-out already holds them
  cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  const uint32_t grid = (p.n_streams + p.lanes_per_warp - 1) / p.lanes_per_warp;
  k<<<grid, 32, smem_bytes, st>>>(a.in, p.d_streams, p.d_order, p.n_streams, p.lanes_per_warp, geom_of(p), a.out, a.dbg,
                                  a.aux, a.tab, p.dump | no_split_bit());
  return cudaGetLastError();
}

template <int NCP, typename T>
static cudaError_t launch_raw_n(const RansLaunch &p, bool table_global, const DevArenas &a, cudaStream_t st) {
  const bool dump = p.dump != 0;
  if (table_global)
    return dump ? launch_raw_t<NCP, T, true, true, 0>(p, a, st) : launch_raw_t<NCP, T, false, true, 0>(p, a, st);
  return dump ? launch_raw_t<NCP, T, true, false, 0>(p, a, st) : launch_raw_t<NCP, T, false, false, 0>(p, a, st);
}

cudaError_t dcb_launch_rans_raw(const RansLaunch &p, int ncp, bool wide, bool table_global, const DevArenas &a,
                                cudaStream_t st) {
#ifdef DCB_DEV_ONLY_C2  // development builds (SASS inspection of the headline instantiation alone): never shipped
  return launch_raw_t<3, uint16_t, false, false, 1, 2, kLeanGroup>(p, a, st);
#else
  // specialised hot shapes (u16 tables in shared memory, no debug dump); compact tables may take the lean loop
  if (!wide && !table_global && !p.dump) {
#define DCB_SPEC(M, N)                                                                           \
  if (p.mode == M && ncp == N) {                                                                 \
    if (!p.compact) return launch_raw_t<N, uint16_t, false, false, M, 1>(p, a, st);              \
    switch (lean_group()) {                                                                      \
      case 4: return launch_raw_t<N, uint16_t, false, false, M, 2, 4>(p, a, st);                 \
      case 16: return launch_raw_t<N, uint16_t, false, false, M, 2, 16>(p, a, st);               \
      default: return launch_raw_t<N, uint16_t, false, false, M, 2, 8>(p, a, st);                \
    }                                                                                            \
  }
    DCB_SPEC(1, 3)
    DCB_SPEC(1, 2)
    DCB_SPEC(2, 3)
    DCB_SPEC(2, 4)
    DCB_SPEC(3, 2)
    DCB_SPEC(4, 3)
    DCB_SPEC(4, 2)
#undef DCB_SPEC
  }
#define DCB_CASE(N)                                                       \
  case N:                                                                 \
    return wide ? launch_raw_n<N, uint32_t>(p, table_global, a, st)       \
                : launch_raw_n<N, uint16_t>(p, table_global, a, st);
  switch (ncp) {
    DCB_CASE(1)
    DCB_CASE(2)
    DCB_CASE(3)
    DCB_CASE(4)
    default:
      return cudaErrorInvalidValue;
  }
#undef DCB_CASE
#endif
}

cudaError_t dcb_launch_rans_tag(const RansLaunch &p, const DevArenas &a, cudaStream_t st) {
  const uint32_t smem_bytes = dcb_rans_smem_bytes(p, false);
  if (smem_bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(rans_tag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (e != cudaSuccess) return e;
  }
  cudaFuncSetAttribute(rans_tag_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  const uint32_t grid = (p.n_streams + p.lanes_per_warp - 1) / p.lanes_per_warp;
  rans_tag_kernel<<<grid, 32, smem_bytes, st>>>(a.in, p.d_streams, p.d_order, p.n_streams, p.lanes_per_warp, geom_of(p),
                                                a.aux);
  return cudaGetLastError();
}

cudaError_t dcb_launch_wide_post(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t dump, const DevArenas &a,
                                 cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  const uint32_t grid = (n + 31) / 32;
  if (dump)
    wide_post_kernel<true><<<grid, 32, 0, st>>>(a.in, d_streams, d_order, n, a.out, a.dbg, a.aux, dump);
  else
    wide_post_kernel<false><<<grid, 32, 0, st>>>(a.in, d_streams, d_order, n, a.out, a.dbg, a.aux, dump);
  return cudaGetLastError();
}

cudaError_t dcb_launch_resolve(const DevArenas &a, BufWalk *d_walks, const uint32_t *d_list, uint32_t n,
                               StreamDesc *d_streams, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  resolve_kernel<<<(n + 63) / 64, 64, 0, st>>>(a.in, d_walks, d_list, n, d_streams);
  return cudaGetLastError();
}

cudaError_t dcb_launch_serial_post(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, int ncp, uint32_t dump,
                                   uint32_t only_irregular, const DevArenas &a, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  const uint32_t grid = (n + 31) / 32;
#define DCB_CASE(N)                                                                                              \
  case N:                                                                                                        \
    if (dump)                                                                                                    \
      serial_post_kernel<N, true><<<grid, 32, 0, st>>>(a.in, d_streams, d_order, n, a.out, a.dbg, a.aux, dump, only_irregular);  \
    else                                                                                                         \
      serial_post_kernel<N, false><<<grid, 32, 0, st>>>(a.in, d_streams, d_order, n, a.out, a.dbg, a.aux, dump, only_irregular); \
    break;
  switch (ncp) {
    DCB_CASE(1)
    DCB_CASE(2)
    DCB_CASE(3)
    DCB_CASE(4)
    default:
      return cudaErrorInvalidValue;
  }
#undef DCB_CASE
  return cudaGetLastError();
}

cudaError_t dcb_launch_para(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, int ncp, uint32_t max_entries,
                            uint32_t dump, const DevArenas &a, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  uint32_t gx = (max_entries + 255) / 256;
  gx = gx < 1 ? 1 : (gx > 1024 ? 1024 : gx);
  para_deps_kernel<<<dim3(gx, n > 65535u ? 65535u : n), 256, 0, st>>>(d_streams, d_order, n, a.maps, a.aux);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const uint32_t grid = n < 148u * 32u ? n : 148u * 32u;  // one warp per stream
#define DCB_CASE(N)                                                                                     \
  case N:                                                                                               \
    if (dump)                                                                                           \
      para_chain_kernel<N, true><<<grid, 64, 0, st>>>(d_streams, d_order, n, a.out, a.dbg, a.aux, dump);  \
    else                                                                                                \
      para_chain_kernel<N, false><<<grid, 64, 0, st>>>(d_streams, d_order, n, a.out, a.dbg, a.aux, dump); \
    break;
  switch (ncp) {
    DCB_CASE(1)
    DCB_CASE(2)
    DCB_CASE(3)
    DCB_CASE(4)
    default:
      return cudaErrorInvalidValue;
  }
#undef DCB_CASE
  return cudaGetLastError();
}

// Kernels that run next to the rANS kernels (side streams) must ask for the same shared-memory carve-out: an SM
// cannot hold CTAs of two carve-out configurations at once, it would drain first.
template <typename K>
static void same_carveout(K k) {
  cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}

cudaError_t dcb_launch_oct_chain(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t dump,
                                 const DevArenas &a, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  const uint32_t grid = (n + 31) / 32;
  same_carveout(oct_chain_kernel<true>);
  same_carveout(oct_chain_kernel<false>);
  if (dump)
    oct_chain_kernel<true><<<grid, 32, 0, st>>>(d_streams, d_order, n, a.aux, a.dbg, dump);
  else
    oct_chain_kernel<false><<<grid, 32, 0, st>>>(d_streams, d_order, n, a.aux, a.dbg, dump);
  return cudaGetLastError();
}

cudaError_t dcb_launch_oct_unit(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint32_t max_entries,
                                const DevArenas &a, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  uint32_t gx = (max_entries + 255) / 256;
  gx = gx < 1 ? 1 : (gx > 4096 ? 4096 : gx);
  same_carveout(oct_unit_kernel);
  oct_unit_kernel<<<dim3(gx, n > 65535u ? 65535u : n), 256, 0, st>>>(d_streams, d_order, n, a.out, a.aux);
  return cudaGetLastError();
}

cudaError_t dcb_launch_copy(StreamDesc *d_streams, const uint32_t *d_order, uint32_t n, uint64_t max_bytes,
                            const DevArenas &a, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  uint64_t gx = (max_bytes + 255) / 256;
  gx = gx < 1 ? 1 : (gx > 2048 ? 2048 : gx);
  copy_kernel<<<dim3((uint32_t)gx, n > 65535u ? 65535u : n), 256, 0, st>>>(a.in, d_streams, d_order, n, a.out);
  return cudaGetLastError();
}
