// draco_sharp_b200/csrc/dcb_rans_pc.cu -- the lane-per-stream rANS kernels as warp PAIRS: a chain warp and a consumer warp.
//
// A rANS stream is one serial chain  x -> slot -> table entry -> x'  (RAnsDecoder.cs:56-67, 90-99); the batch time is
// (symbols per stream) x (cycles per chain step).  A warp issues in order, so everything else that shares the warp
// with the chain -- value map, zig-zag, delta + wrap, dequantisation, the stores -- sits between two chain
// instructions and stretches the step (round 1: 69 instructions and 178 cycles per symbol for a chain whose own
// dependent latency is ~105 cycles).  Here the two halves live in different warps of one CTA:
//
//   chain warp     lane l runs stream l's chain and nothing else: renormalise, two-region LUT probe, state update,
//                  and ONE 16-bit store per symbol (the table-entry offset) into a shared-memory queue.
//   consumer warp  lane l pops stream l's entry offsets one group (4 entries) behind the chain and does what
//                  SequentialIntegerAttributeDecoder.DecodeIntegerValues does after DecodeSymbols (:86-101): value map
//                  / zig-zag (BitUtilities.cs:72-81), PredictionSchemeDeltaDecoder + wrap transform
//                  (PredictionSchemeWrapDecodingTransform.cs:46-67), dequantisation (Dequantizer.cs:14-23) or the
//                  narrowing store (:142-160), 128-bit stores.
//
// The queue is kStages groups deep; its rows are lane-interleaved (row j holds symbol j of every lane, 2 bytes per
// lane), so neither side ever has a bank conflict on it.  Hand-over is by mbarrier: full[s] (chain -> consumer) and
// empty[s] (consumer -> chain), one arrival each by an elected lane after __syncwarp.  The chain warp never blocks on
// empty[s] in steady state: it TESTS the barrier of group g+1 (non-blocking) while it decodes group g and only
// looks at the answer a group later.
//
// A CTA holds `pairs` such pairs (warps 0..pairs-1 are chain warps, pairs..2*pairs-1 their consumers), each with its
// own slice of shared memory, so that with four pairs every SM sub-partition runs one chain and one consumer warp.
//
// Exactness at the ends of a stream is unchanged from round 1: the queue carries the warp-uniform main loop only
// (groups every lane can decode without running out of bytes); then the consumer hands its running values back and
// the chain warp itself finishes each stream with the careful per-entry loop (`off > 0` checked per byte).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <algorithm>

#include "dcb_device.cuh"
#include "dcb_internal.h"
#include "dcb_kernels.h"

using namespace dcb;

namespace {

constexpr uint32_t kStages = DCB_PC_STAGES;      // queue depth in groups (power of two)
constexpr uint32_t kRowBytes = DCB_PC_ROW_BYTES; // one queue row: 32 lanes x 2 bytes

// what the two warps of a pair tell each other outside the queue, per lane
struct LaneHand {
  uint32_t dprefix;     // chain -> consumer: dense prefix of the lane's compact table (RansLane::dprefix)
  int32_t active;       // chain -> consumer: the lane decodes a stream (tables built, state initialised)
  int32_t prev[4];      // consumer -> chain: running values of the delta decoder after the last queued group
  int32_t status;       // tags: consumer -> chain
  uint32_t e;           // tags: consumer -> chain: first tag the careful tail has to decode
  uint32_t ne;          // chain -> both: table entries built (direct slot LUT fill)
  uint32_t fused;       // chain -> consumer (first record of the slice): the chain warp runs the fused main loop, leave
  uint64_t bits;        // tags: consumer -> chain: bits consumed in the bit area so far
};
static_assert(sizeof(LaneHand) == DCB_PC_HAND_BYTES, "LaneHand size is part of the shared-memory plan");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t a, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(a), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t a) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(a) : "memory");
}
// non-blocking: has the phase with this parity completed?
__device__ __forceinline__ uint32_t mbar_test(uint32_t a, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(a), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait(uint32_t a, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "PC_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra PC_DONE;\n"
      "bra PC_WAIT;\n"
      "PC_DONE:\n"
      "}\n" ::"r"(a),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void sts_u16(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u16 [%0], %1;\n" ::"r"(a), "h"((uint16_t)v) : "memory");
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;\n" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u16 %0, [%1];\n" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t lds_u32m(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(a) : "memory");
  return v;
}

// addresses of a pair's control block (DCB_PC_CTL_BYTES): full[kStages] | empty[kStages] | setup | handoff | filled | flag[kStages]
constexpr uint32_t kNumBarriers = 2u * kStages + 3u;
struct PairCtl {
  uint32_t base;
  __device__ __forceinline__ uint32_t full(uint32_t s) const { return base + 8u * s; }
  __device__ __forceinline__ uint32_t empty(uint32_t s) const { return base + 8u * (kStages + s); }
  __device__ __forceinline__ uint32_t setup() const { return base + 16u * kStages; }
  __device__ __forceinline__ uint32_t handoff() const { return base + 16u * kStages + 8u; }
  __device__ __forceinline__ uint32_t filled() const { return base + 16u * kStages + 16u; }  // two arrivals: both warps
  __device__ __forceinline__ uint32_t flag(uint32_t s) const { return base + 8u * kNumBarriers + 4u * s; }
};
static_assert(8u * kNumBarriers + 4u * kStages <= DCB_PC_CTL_BYTES, "control block");

// Direct slot LUT of one lane, filled by both warps of the pair (64 threads): for every slot the table entry that owns
// it -- what RAnsDecoder.BuildLookupTable (RAnsDecoder.cs:69-88) materialises as lut[] -- folded with that entry's
// frequency and the slot's offset inside it, so that the chain needs ONE dependent shared-memory access per symbol.
__device__ __forceinline__ void fill_direct(const uint16_t *cum, uint32_t ne, uint32_t prec_bits, uint32_t ent_off,
                                            uint16_t *freq, uint16_t *off, uint16_t *ent, uint32_t tid, uint32_t nthreads) {
  const uint32_t n = 1u << prec_bits;
  for (uint32_t s = tid; s < n; s += nthreads) {
    uint32_t lo = 0, hi = ne;  // cum[lo] <= s; hi == ne or cum[hi] > s  (zero-width entries of dense tables: the last one wins)
    while (hi - lo > 1u) {
      const uint32_t mid = (lo + hi) >> 1;
      if ((uint32_t)cum[mid] <= s) lo = mid;
      else hi = mid;
    }
    const uint32_t c = cum[lo];
    freq[s] = (uint16_t)((uint32_t)cum[lo + 1] - c);
    off[s] = (uint16_t)(s - c);
    ent[s] = (uint16_t)(ent_off + 2u * lo);
  }
}
// both warps of a pair, after the chain warp has built the tables: fill every active lane's direct LUT, then meet
__device__ __forceinline__ void fill_direct_all(uint8_t *slice, const SmemLayout &lay, const TableGeom &geom, uint32_t lanes,
                                                uint32_t hand_off, uint32_t prec_bits, uint32_t tid64, const PairCtl &ctl) {
  const uint32_t arr = 2u << prec_bits;  // bytes of one u16 array
  for (uint32_t l = 0; l < lanes; ++l) {
    const volatile uint32_t *h = reinterpret_cast<const volatile uint32_t *>(slice + hand_off + (size_t)l * DCB_PC_HAND_BYTES);
    if (h[1] == 0u) continue;  // LaneHand::active
    const uint32_t ne = h[8];  // LaneHand::ne
    uint8_t *lut = slice + lay.lut0 + (size_t)l * geom.lut_bytes;
    fill_direct(reinterpret_cast<const uint16_t *>(slice + lay.ent0 + (size_t)l * geom.ent_bytes), ne, prec_bits, l * geom.ent_bytes,
                reinterpret_cast<uint16_t *>(lut), reinterpret_cast<uint16_t *>(lut + arr), reinterpret_cast<uint16_t *>(lut + 2u * arr),
                tid64, 64u);
  }
  __syncwarp();
  if ((tid64 & 31u) == 0u) mbar_arrive(ctl.filled());
  mbar_wait(ctl.filled(), 0u);
}

// Which pair a warp belongs to and on which side.  Packed layout: warps 0..pairs-1 are chain warps, the next `pairs`
// their consumers (a pair shares a sub-partition when pairs == 4).  Split layout (bit 31 of `pairs`, at most 3 pairs,
// 4 * pairs warps): chain warps 0..pairs-1 have a sub-partition each to themselves (warp id mod 4), ALL consumers sit
// on sub-partition 3 (warps 3, 7, 11), the warps in between leave at once.  The ALU and FMA pipes of a sub-partition
// take one warp instruction every two cycles each, so a consumer next to its chain warp takes issue slots from it.
__device__ __forceinline__ void warp_role(uint32_t warp, uint32_t &pairs, uint32_t &pair, uint32_t &role) {
  const bool split = (pairs >> 31) != 0u, chain_low = ((pairs >> 30) & 1u) != 0u;
  pairs &= 0x3FFFFFFFu;
  if (!split) {
    // the sub-partition's arbiter prefers the warp with the higher id: the chain warps take the upper half, so that
    // the consumer only gets the issue slots the chain leaves
    pair = warp % pairs;
    role = chain_low ? warp / pairs : 1u - warp / pairs;
  } else if (warp < pairs) {
    pair = warp;
    role = 0;
  } else if ((warp & 3u) == 3u) {
    pair = warp >> 2;
    role = 1;
  } else {
    pair = 0;
    role = 2;
  }
}

// The chain warp's main loop.  NSYM symbols per group and lane; returns the number of groups queued.
// `go0`: the warp has at least one full group that every active lane can decode without byte-bound checks.
template <int NSYM, int PROBE>
__device__ __forceinline__ uint32_t produce(RansLane<uint16_t, false> &rl, bool active, uint32_t g_min, uint32_t q_addr,
                                            const PairCtl &ctl, uint32_t lane) {
  constexpr uint32_t kGroupBytes = (uint32_t)NSYM * 3u;
  uint32_t g = 0;
  bool go = g_min != 0xFFFFFFFFu && g_min > 0u && __all_sync(0xffffffffu, !active || rl.bytes_left() >= kGroupBytes);
  uint32_t slot_free = 1u;  // the first kStages groups find their slots untouched
  while (go) {
    const uint32_t s = g & (kStages - 1u), par = (g / kStages) & 1u;
    if (!slot_free) mbar_wait(ctl.empty(s), par ^ 1u);
    {
      const uint32_t g1 = g + 1u;
      slot_free = mbar_test(ctl.empty(g1 & (kStages - 1u)), ((g1 / kStages) & 1u) ^ 1u);
    }
    const uint32_t qs = q_addr + s * ((uint32_t)NSYM * kRowBytes) + lane * 2u;
    if (active) {
#pragma unroll
      for (int j = 0; j < NSYM; ++j) {
        const uint32_t o = PROBE == 2 ? rl.step_direct_slot() : rl.template step<false, PROBE>();
        sts_u16(qs + (uint32_t)j * kRowBytes, o);
      }
    }
    const bool next_go = (g + 1u < g_min) && __all_sync(0xffffffffu, !active || rl.bytes_left() >= kGroupBytes);
    if (active) {
      rl.template top_up<(kGroupBytes + 15) / 16 + 1>();
      cp_async_wait<1>();
    }
    __syncwarp();
    if (lane == 0) {
      sts_u32(ctl.flag(s), 0u);
      mbar_arrive(ctl.full(s));
    }
    ++g;
    go = next_go;
  }
  {  // end marker: the consumer hands its running values back and the chain warp finishes every stream itself
    const uint32_t s = g & (kStages - 1u), par = (g / kStages) & 1u;
    if (!slot_free) mbar_wait(ctl.empty(s), par ^ 1u);
    __syncwarp();
    if (lane == 0) {
      sts_u32(ctl.flag(s), 1u);
      mbar_arrive(ctl.full(s));
    }
  }
  return g;
}

// table entry offset -> symbol value, for the consumer warp (RansLane::value without the chain's state)
struct ValMap {
  const uint8_t *ent0;
  uint32_t ent_off, dprefix, val_delta;
  __device__ __forceinline__ int32_t value(uint32_t o, bool compact, bool zig) const {
    const uint32_t rank = (o - ent_off) >> 1;
    if (compact && rank >= dprefix) {
      return zig ? (int32_t) * reinterpret_cast<const int16_t *>(ent0 + o + val_delta)
                 : (int32_t) * reinterpret_cast<const uint16_t *>(ent0 + o + val_delta);
    }
    return zig ? zigzag_dec(rank) : (int32_t)rank;
  }
  __device__ __forceinline__ uint32_t symbol(uint32_t o, bool compact, bool zig) const {
    const int32_t v = value(o, compact, zig);
    if (!zig) return (uint32_t)v;
    return v >= 0 ? ((uint32_t)v << 1) : ((((uint32_t)(-(v + 1))) << 1) | 1u);
  }
};

// launch-wide redirections of the post-processing (same rules as rans_raw_fused_kernel)
template <int NCP, int MODE>
__device__ __forceinline__ void redirect_post(PostParams &pp, uint32_t &dump, uint8_t *&optr, uint8_t *aux, const StreamDesc &d) {
  if (MODE == 3 || MODE == 4 || (MODE == 0 && (pp.recon == RECON_PARA_WRAP || pp.store == STORE_OCT_UNIT))) {
    optr = aux + d.aux_off;  // int32 scratch: corrections for the parallelogram kernel / for oct_chain_kernel
    if (NCP == 2 && pp.store == STORE_OCT_UNIT) {
      pp.recon = RECON_NONE;
      dump &= ~(uint32_t)DCB_DUMP_QINTS;
    }
    pp.store = STORE_NARROW;
    pp.dsize = 4;
  }
}

// ---------------------------------------------------------------------------------------------
// Raw scheme (SymbolDecoding.cs:52-67) fused with inverse prediction + transform + store
// ---------------------------------------------------------------------------------------------
// FUSED main loop on the direct slot LUT: the chain warp keeps the post-processing and runs the software-pipelined lean
// loop of dcb_device.cuh (lean_sp_group, one dependent LDS per symbol, the previous symbol's value map / wrap / store
// in its latency shadow).  With a handful of lanes per warp the queue push costs the chain about what the
// post-processing does, and the consumer warp shares the sub-partition's issue port.  Returns the groups decoded.
template <int NCP, int MODE, bool COMPACT>
__device__ __forceinline__ uint32_t fused_direct_loop(RansLane<uint16_t, false> &rl, const PostParams &pp, uint8_t *optr,
                                                      uint32_t g_min, int32_t *prev, uint32_t zero) {
  constexpr uint32_t kGroupBytes = 4u * NCP * 3u;
  uint32_t g = 0;
  if (g_min != 0xFFFFFFFFu && g_min > 0 && rl.bytes_left() >= kGroupBytes) {
    rl.window_open();  // prologue: symbol 0 of group 0
    uint32_t ca_prev = rl.template step_lean_direct<true>(0u, zero);
    uint32_t gate = 0;
    while (g + 1 < g_min && rl.bytes_left() >= 2u * kGroupBytes + 4u) {
      lean_sp_group<NCP, MODE, false, 2, COMPACT>(rl, pp, optr, g, prev, ca_prev, gate, zero);  // tops the ring up
      ++g;
    }
    lean_sp_group<NCP, MODE, true, 2, COMPACT>(rl, pp, optr, g, prev, ca_prev, gate, zero);
    ++g;
    cp_async_wait<1>();
  }
  rl.prefetch();  // the careful tail reads through the two-word peek
  return g;
}

template <int NCP, bool DUMP, int MODE, int TAB>
__global__ void __launch_bounds__(384) rans_raw_pc_kernel(const uint8_t *__restrict__ arena, StreamDesc *streams,
                                                          const uint32_t *__restrict__ order, uint32_t n_streams,
                                                          uint32_t lanes, uint32_t pairs, TableGeom geom, PcGeom pc,
                                                          uint8_t *__restrict__ out, uint8_t *__restrict__ dbg,
                                                          uint8_t *__restrict__ aux, uint32_t dump) {
  extern __shared__ __align__(16) uint8_t smem[];
  typedef uint16_t T;
  constexpr int kSym = 4 * NCP;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t pair, role;
  warp_role(warp, pairs, pair, role);
  uint8_t *slice = smem + (size_t)pair * pc.slice_bytes;
  const uint32_t slice_addr = smem_u32(slice);
  const uint32_t q_addr = slice_addr + pc.q_off;
  const PairCtl ctl{slice_addr + pc.ctl_off};
  if (role == 0 && lane == 0) {
#pragma unroll
    for (uint32_t i = 0; i < kNumBarriers; ++i) mbar_init(ctl.base + 8u * i, i == 2u * kStages + 2u ? 2u : 1u);
  }
  __syncthreads();
  if (role == 2u) return;
  const uint32_t slot = (blockIdx.x * pairs + pair) * lanes + lane;
  const bool have = lane < lanes && slot < n_streams;
  StreamDesc *dp = have ? &streams[order[slot]] : nullptr;
  LaneHand *hand = reinterpret_cast<LaneHand *>(slice + pc.hand_off) + (have ? lane : 0u);
  const SmemLayout lay = smem_layout(slice_addr, lanes, geom, false);
  const bool compact = TAB == 0 ? geom.compact != 0 : TAB == 2;
  const bool zig = MODE == 0 ? geom.zig != 0 : MODE != 3;

  if (role == 0) {
    // ================================ chain warp ================================
    RansLane<T, false> rl;
    uint32_t n_entries = 0;
    bool split_ok = true;  // idle lanes do not veto
    T *lut = nullptr, *ent = nullptr;
    uint8_t *lutb = nullptr;
    uint32_t *blk = nullptr;
    rl.dprefix = 0;
    if (have) {
      const StreamDesc &d = *dp;
      n_entries = d.n_entries;
      int status = DCB_OK;
      if (n_entries > 0) {
        rl.lut0 = nullptr;
        rl.ent0 = slice + lay.ent0;
        rl.lut_base = slice_addr + lay.lut0 + lane * geom.lut_bytes;
        rl.lutb_addr = slice_addr + lay.lutb0 + lane * geom.lutb_bytes;
        rl.blk_addr = slice_addr + lay.blk0 + lane * geom.blk_bytes;
        blk = reinterpret_cast<uint32_t *>(slice + lay.blk0 + (size_t)lane * geom.blk_bytes);
        const uint32_t ent_off = lane * geom.ent_bytes;
        rl.cum_addr = slice_addr + lay.ent0 + ent_off;
        lut = reinterpret_cast<T *>(slice + lay.lut0 + (size_t)lane * geom.lut_bytes);
        lutb = slice + lay.lutb0 + (size_t)lane * geom.lutb_bytes;
        ent = reinterpret_cast<T *>(slice + lay.ent0 + (size_t)lane * geom.ent_bytes);
        if (geom.direct) {
          rl.d_freq = slice_addr + lay.lut0 + lane * geom.lut_bytes;
          rl.d_off = rl.d_freq + (2u << d.prec_bits);
          rl.d_ent = rl.d_off + (2u << d.prec_bits);
        }
        status = rl.build(arena, d, geom, ent, ent_off);
        if (status == DCB_OK) status = rl.init_state(arena, d);
        if (status == DCB_OK) split_ok = rl.split_ok && !(dump & 0x80000000u);
      }
      if (status != DCB_OK) {
        dp->status = status;
        n_entries = 0;
      }
    }
    const bool use_split = __all_sync(0xffffffffu, split_ok);
    const bool active = n_entries > 0;
    uint32_t g_min = active ? (n_entries >> 2) : 0xFFFFFFFFu;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) g_min = min(g_min, __shfl_xor_sync(0xffffffffu, g_min, o));
    if (active) {
      if (!geom.direct) rl.fill_lut(geom, lut, lutb, blk, ent, use_split);
      rl.init_ring(slice_addr + lay.ring0 + lane * DCB_RING_BYTES);
    }
    if (have) {
      hand->dprefix = rl.dprefix;
      hand->active = active ? 1 : 0;
      hand->ne = active ? rl.n_entries_tab : 0u;
    }
    // fused main loop (fused_direct_loop): direct slot LUT, zig-zag coded corrections of a specialised mode, no dumps;
    // delta + wrap modes only on regular streams (wrap_regular, as the lean loop of rans_raw_fused_kernel)
    bool fuse_ok = true;
    constexpr bool kFusable = !DUMP && MODE >= 1 && MODE <= 4 && TAB != 0;
    if (kFusable && active && (MODE == 1 || MODE == 2)) {
      const int64_t md = 1ll + (int64_t)dp->xf_b - (int64_t)dp->xf_a;
      fuse_ok = (int64_t)rl.max_abs_val < md && dp->xf_a >= -(1 << 29) && dp->xf_b <= (1 << 29);
    }
    const bool fuse = kFusable && zig && geom.zig != 0u && geom.direct && pc.fuse != 0u && __all_sync(0xffffffffu, fuse_ok);
    if (lane == 0) reinterpret_cast<LaneHand *>(slice + pc.hand_off)->fused = fuse ? 1u : 0u;
    __syncwarp();
    if (lane == 0) mbar_arrive(ctl.setup());
    const int probe = geom.direct ? 2 : (use_split ? 1 : 0);
    if (geom.direct) {
      mbar_wait(ctl.setup(), 0u);
      fill_direct_all(slice, lay, geom, lanes, pc.hand_off, geom.direct_prec, lane, ctl);
    }
    PostParams pp;
    uint8_t *optr = nullptr;
    int32_t *dptr = nullptr;
    if (active) {
      pp.load(*dp);
      optr = out + dp->out_off;
      dptr = DUMP ? reinterpret_cast<int32_t *>(dbg + dp->dbg_off) : nullptr;
      redirect_post<NCP, MODE>(pp, dump, optr, aux, *dp);
    }
    int32_t prev[NCP];
    uint32_t groups = 0;
    if (fuse) {
      if (!active) return;
      const int32_t p0 = (MODE == 1 || MODE == 2) ? (0 > pp.mx ? pp.mx : (0 < pp.mn ? pp.mn : 0)) : 0;
#pragma unroll
      for (int c = 0; c < NCP; ++c) prev[c] = p0;
      if constexpr (kFusable) groups = fused_direct_loop<NCP, MODE, TAB == 2>(rl, pp, optr, g_min, prev, blockIdx.y);
    } else {
      groups = probe == 2 ? produce<kSym, 2>(rl, active, g_min, q_addr, ctl, lane)
             : probe == 1 ? produce<kSym, 1>(rl, active, g_min, q_addr, ctl, lane)
                          : produce<kSym, 0>(rl, active, g_min, q_addr, ctl, lane);
      mbar_wait(ctl.handoff(), 0u);
      if (!active) return;
#pragma unroll
      for (int c = 0; c < NCP; ++c) prev[c] = hand->prev[c];
    }
    // ---- per-lane tail: exact `off > 0` handling, as RAnsDecoder.Read does it byte by byte ----
    const int store = store_of<MODE>(pp), dsize = dsize_of<MODE>(pp);
    for (uint32_t e = groups * 4u; e < n_entries; ++e) {
      int32_t v[NCP];
      if (probe == 2) decode_entry<NCP, T, false, DUMP, MODE, TAB, true, 2>(rl, geom, pp, prev, v, dptr, dump, e);
      else if (probe == 1) decode_entry<NCP, T, false, DUMP, MODE, TAB, true, 1>(rl, geom, pp, prev, v, dptr, dump, e);
      else decode_entry<NCP, T, false, DUMP, MODE, TAB, true, 0>(rl, geom, pp, prev, v, dptr, dump, e);
      store_entry<NCP>(pp, store, dsize, optr, e, v);
      rl.template top_up<(3 * NCP + 15) / 16 + 1>();
      cp_async_wait<0>();
    }
  } else {
    // ================================ consumer warp ================================
    PostParams pp;
    uint8_t *optr = nullptr;
    int32_t *dptr = nullptr;
    if (have) {
      pp.load(*dp);
      optr = out + dp->out_off;
      dptr = DUMP ? reinterpret_cast<int32_t *>(dbg + dp->dbg_off) : nullptr;
      redirect_post<NCP, MODE>(pp, dump, optr, aux, *dp);
    }
    const int store = store_of<MODE>(pp), dsize = dsize_of<MODE>(pp), recon = recon_of<MODE>(pp);
    mbar_wait(ctl.setup(), 0u);
    if (geom.direct) fill_direct_all(slice, lay, geom, lanes, pc.hand_off, geom.direct_prec, 32u + lane, ctl);
    if (reinterpret_cast<const volatile LaneHand *>(slice + pc.hand_off)->fused != 0u) return;  // the chain warp does it all
    const uint32_t d_ent = slice_addr + lay.lut0 + lane * geom.lut_bytes + (4u << geom.direct_prec);  // direct LUT: entry[] of this lane
    bool active = false;
    ValMap vm{slice + lay.ent0, lane * geom.ent_bytes, 0u, 0u};
    if (have) {
      active = hand->active != 0;
      vm.dprefix = hand->dprefix;
      vm.val_delta = (geom.cap_entries + 2u - (geom.compact ? vm.dprefix : 0u)) * 2u;
    }
    int32_t prev[NCP];
#pragma unroll
    for (int c = 0; c < NCP; ++c) prev[c] = 0;
    for (uint32_t g = 0;; ++g) {
      const uint32_t s = g & (kStages - 1u);
      mbar_wait(ctl.full(s), (g / kStages) & 1u);
      if (lds_u32m(ctl.flag(s)) != 0u) break;
      const uint32_t qs = q_addr + s * ((uint32_t)kSym * kRowBytes) + lane * 2u;
      int32_t v[4][NCP];
      if (active) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int c = 0; c < NCP; ++c) {
            uint32_t o = lds_u16(qs + (uint32_t)(j * NCP + c) * kRowBytes);
            if (geom.direct) o = lds_u16(d_ent + 2u * o);  // the chain queued the slot
            v[j][c] = vm.value(o, compact, zig);
            if (DUMP && (dump & DCB_DUMP_SYMBOLS)) dptr[((uint64_t)g * 4 + j) * NCP + c] = (int32_t)vm.symbol(o, compact, zig);
          }
      }
      // every queued offset of this group is in registers (the value map consumed it): the slot may be refilled
      __syncwarp();
      if (lane == 0) mbar_arrive(ctl.empty(s));
      if (active) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (recon == RECON_DELTA_WRAP) {
#pragma unroll
            for (int c = 0; c < NCP; ++c) {
              prev[c] = wrap_original(prev[c], v[j][c], pp.mn, pp.mx, pp.max_diff);
              v[j][c] = prev[c];
            }
          } else if (recon == RECON_DELTA_OCT || recon == RECON_DELTA_OCT_CANON) {
            if (NCP == 2) {
              oct_original(pp.box, recon == RECON_DELTA_OCT_CANON, prev[0], prev[NCP - 1], v[j][0], v[j][NCP - 1]);
              v[j][0] = prev[0];
              v[j][NCP - 1] = prev[NCP - 1];
            }
          }
          if (DUMP && MODE != 3 && (dump & DCB_DUMP_QINTS)) {
#pragma unroll
            for (int c = 0; c < NCP; ++c) dptr[((uint64_t)g * 4 + j) * NCP + c] = v[j][c];
          }
        }
        store_group4<NCP>(pp, store, dsize, optr, (uint64_t)g * 4, v);
      }
    }
    if (have) {
#pragma unroll
      for (int c = 0; c < NCP; ++c) hand->prev[c] = prev[c];
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(ctl.handoff());
  }
}

// ---------------------------------------------------------------------------------------------
// Tag stream of a Tagged attribute (SymbolDecoding.cs:30-50): one rANS symbol per point = the bit length of its
// values.  Chain warp as above, 16 tags per group; the consumer writes one byte per point, the running bit
// offset at every DCB_TAG_CHUNK points and validates (tag <= 32, DecoderBuffer.cs:141; bit area inside the buffer).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(384) rans_tag_pc_kernel(const uint8_t *__restrict__ arena, StreamDesc *streams,
                                                          const uint32_t *__restrict__ order, uint32_t n_streams,
                                                          uint32_t lanes, uint32_t pairs, TableGeom geom, PcGeom pc,
                                                          uint8_t *__restrict__ aux) {
  extern __shared__ __align__(16) uint8_t smem[];
  typedef uint16_t T;
  constexpr int kSym = 16;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t pair, role;
  warp_role(warp, pairs, pair, role);
  uint8_t *slice = smem + (size_t)pair * pc.slice_bytes;
  const uint32_t slice_addr = smem_u32(slice);
  const uint32_t q_addr = slice_addr + pc.q_off;
  const PairCtl ctl{slice_addr + pc.ctl_off};
  if (role == 0 && lane == 0) {
#pragma unroll
    for (uint32_t i = 0; i < kNumBarriers; ++i) mbar_init(ctl.base + 8u * i, i == 2u * kStages + 2u ? 2u : 1u);
  }
  __syncthreads();
  if (role == 2u) return;
  const uint32_t slot = (blockIdx.x * pairs + pair) * lanes + lane;
  const bool have = lane < lanes && slot < n_streams;
  StreamDesc *dp = have ? &streams[order[slot]] : nullptr;
  LaneHand *hand = reinterpret_cast<LaneHand *>(slice + pc.hand_off) + (have ? lane : 0u);
  const SmemLayout lay = smem_layout(slice_addr, lanes, geom, false);
  const bool compact = geom.compact != 0;

  if (role == 0) {
    RansLane<T, false> rl;
    T *ent = reinterpret_cast<T *>(slice + lay.ent0 + (size_t)lane * geom.ent_bytes);
    bool active = false, split_ok = true;
    rl.dprefix = 0;
    if (have) {
      rl.lut0 = nullptr;
      rl.ent0 = slice + lay.ent0;
      rl.lut_base = slice_addr + lay.lut0 + lane * geom.lut_bytes;
      rl.lutb_addr = slice_addr + lay.lutb0 + lane * geom.lutb_bytes;
      rl.blk_addr = slice_addr + lay.blk0 + lane * geom.blk_bytes;
      rl.cum_addr = slice_addr + lay.ent0 + lane * geom.ent_bytes;
      if (geom.direct) {
        rl.d_freq = slice_addr + lay.lut0 + lane * geom.lut_bytes;
        rl.d_off = rl.d_freq + (2u << geom.direct_prec);
        rl.d_ent = rl.d_off + (2u << geom.direct_prec);
      }
      int status = rl.build(arena, *dp, geom, ent, lane * geom.ent_bytes);
      if (status == DCB_OK) status = rl.init_state(arena, *dp);
      if (status != DCB_OK) {
        dp->status = status;
        dp->bits_total = 0;
      } else {
        active = true;
        split_ok = rl.split_ok;
      }
    }
    const bool use_split = __all_sync(0xffffffffu, split_ok);
    const uint32_t n_entries = active ? dp->n_entries : 0u;
    uint32_t g_min = active ? (n_entries >> 4) : 0xFFFFFFFFu;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) g_min = min(g_min, __shfl_xor_sync(0xffffffffu, g_min, o));
    if (active) {
      if (!geom.direct)
        rl.fill_lut(geom, reinterpret_cast<T *>(slice + lay.lut0 + (size_t)lane * geom.lut_bytes),
                    slice + lay.lutb0 + (size_t)lane * geom.lutb_bytes,
                    reinterpret_cast<uint32_t *>(slice + lay.blk0 + (size_t)lane * geom.blk_bytes), ent, use_split);
      rl.init_ring(slice_addr + lay.ring0 + lane * DCB_RING_BYTES);
    }
    if (have) {
      hand->dprefix = rl.dprefix;
      hand->active = active ? 1 : 0;
      hand->ne = active ? rl.n_entries_tab : 0u;
    }
    // fused: the chain warp keeps the (small) post-processing of the tags -- run_tags_sp on the direct slot LUT
    const bool fuse = geom.direct && pc.fuse != 0u;
    if (lane == 0) reinterpret_cast<LaneHand *>(slice + pc.hand_off)->fused = fuse ? 1u : 0u;
    __syncwarp();
    if (lane == 0) mbar_arrive(ctl.setup());
    const int probe = geom.direct ? 2 : (use_split ? 1 : 0);
    if (geom.direct) {
      mbar_wait(ctl.setup(), 0u);
      fill_direct_all(slice, lay, geom, lanes, pc.hand_off, geom.direct_prec, lane, ctl);
    }
    if (fuse) {
      if (active) run_tags_sp<2>(rl, geom, dp, aux, blockIdx.y);  // blockIdx.y: an opaque zero
      return;
    }
    if (probe == 2) produce<kSym, 2>(rl, active, g_min, q_addr, ctl, lane);
    else if (probe == 1) produce<kSym, 1>(rl, active, g_min, q_addr, ctl, lane);
    else produce<kSym, 0>(rl, active, g_min, q_addr, ctl, lane);
    mbar_wait(ctl.handoff(), 0u);
    if (!active) return;
    // ---- careful tail (exact `off > 0` handling, per-point checks) ----
    const StreamDesc &d = *dp;
    const uint32_t ncp = d.ncp;
    const uint64_t avail_bits = (d.buf_end - d.bits_off) * 8ull;
    uint8_t *tags = aux + d.tag_off;
    uint64_t *chunk_bits = reinterpret_cast<uint64_t *>(aux + d.tag_off + (((uint64_t)n_entries + 15ull) & ~15ull));
    int status = hand->status;
    uint64_t bits = hand->bits;
    for (uint32_t e = hand->e; status == DCB_OK && e < n_entries; ++e) {
      if ((e & (DCB_TAG_CHUNK - 1u)) == 0) chunk_bits[e / DCB_TAG_CHUNK] = bits;
      const uint32_t o = probe == 2 ? rl.template step<true, 2>() : probe == 1 ? rl.template step<true, 1>() : rl.template step<true, 0>();
      const uint32_t tag = (uint32_t)rl.value(o, compact, false) & 0xFFu;  // (byte) cast, SymbolDecoding.cs:41
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
      rl.template top_up<1>();
      cp_async_wait<0>();
    }
    dp->bits_total = bits;
    if (status != DCB_OK) dp->status = status;
  } else {
    uint32_t n_entries = 0, ncp = 0;
    uint64_t avail_bits = 0;
    uint8_t *tags = nullptr;
    uint64_t *chunk_bits = nullptr;
    if (have) {
      const StreamDesc &d = *dp;
      n_entries = d.n_entries;
      ncp = d.ncp;
      avail_bits = (d.buf_end - d.bits_off) * 8ull;
      tags = aux + d.tag_off;
      chunk_bits = reinterpret_cast<uint64_t *>(aux + d.tag_off + (((uint64_t)n_entries + 15ull) & ~15ull));
    }
    mbar_wait(ctl.setup(), 0u);
    if (geom.direct) fill_direct_all(slice, lay, geom, lanes, pc.hand_off, geom.direct_prec, 32u + lane, ctl);
    if (reinterpret_cast<const volatile LaneHand *>(slice + pc.hand_off)->fused != 0u) return;  // the chain warp does it all
    const uint32_t d_ent = slice_addr + lay.lut0 + lane * geom.lut_bytes + (4u << geom.direct_prec);
    bool active = false;
    ValMap vm{slice + lay.ent0, lane * geom.ent_bytes, 0u, 0u};
    if (have) {
      active = hand->active != 0;
      vm.dprefix = hand->dprefix;
      vm.val_delta = (geom.cap_entries + 2u - (geom.compact ? vm.dprefix : 0u)) * 2u;
    }
    int status = DCB_OK;
    uint64_t bits = 0;
    uint32_t e = 0;
    for (uint32_t g = 0;; ++g) {
      const uint32_t s = g & (kStages - 1u);
      mbar_wait(ctl.full(s), (g / kStages) & 1u);
      if (lds_u32m(ctl.flag(s)) != 0u) break;
      const uint32_t qs = q_addr + s * ((uint32_t)kSym * kRowBytes) + lane * 2u;
      uint32_t t[16];
      if (active) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          uint32_t o = lds_u16(qs + (uint32_t)j * kRowBytes);
          if (geom.direct) o = lds_u16(d_ent + 2u * o);
          t[j] = (uint32_t)vm.value(o, compact, false) & 0xFFu;  // (byte) cast, SymbolDecoding.cs:41
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(ctl.empty(s));
      if (active && status == DCB_OK) {
        if ((e & (DCB_TAG_CHUNK - 1u)) == 0) chunk_bits[e / DCB_TAG_CHUNK] = bits;
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
        } else {
          uint4 pk;
          pk.x = t[0] | (t[1] << 8) | (t[2] << 16) | (t[3] << 24);
          pk.y = t[4] | (t[5] << 8) | (t[6] << 16) | (t[7] << 24);
          pk.z = t[8] | (t[9] << 8) | (t[10] << 16) | (t[11] << 24);
          pk.w = t[12] | (t[13] << 8) | (t[14] << 16) | (t[15] << 24);
          *reinterpret_cast<uint4 *>(tags + e) = pk;
          bits = nbits;
          e += 16;
        }
      }
    }
    if (have) {
      hand->status = status;
      hand->bits = bits;
      hand->e = e;
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(ctl.handoff());
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static uint32_t chain_low_bit() {  // DCB_CHAIN_LOW=1: chain warps in the lower half of the CTA (experiments)
  static const uint32_t bit = getenv("DCB_CHAIN_LOW") ? 0x40000000u : 0u;
  return bit;
}
static TableGeom pc_table_geom(const RansLaunch &p) {
  TableGeom g{};
  g.direct = p.direct;
  g.direct_prec = p.prec_bits;
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

PcGeom dcb_pc_geom(const RansLaunch &p, uint32_t syms_per_group) {
  PcGeom g;
  g.tab_bytes = (dcb_rans_smem_bytes(p, false) + 15u) & ~15u;
  g.q_off = g.tab_bytes;
  g.ctl_off = g.q_off + DCB_PC_STAGES * syms_per_group * DCB_PC_ROW_BYTES;
  g.hand_off = g.ctl_off + DCB_PC_CTL_BYTES;
  g.slice_bytes = (g.hand_off + p.lanes_per_warp * DCB_PC_HAND_BYTES + 15u) & ~15u;
  static const bool no_fuse = getenv("DCB_NO_PC_FUSED") != nullptr;  // A/B measurements, tests of the queue path
  g.fuse = no_fuse ? 0u : 1u;
  return g;
}

uint32_t dcb_rans_pc_smem_bytes(const RansLaunch &p, uint32_t syms_per_group) {
  return dcb_pc_geom(p, syms_per_group).slice_bytes * std::max(1u, p.pairs);
}

static uint32_t pc_no_split_bit() {
  static const uint32_t bit = getenv("DCB_NO_SPLIT") ? 0x80000000u : 0u;
  return bit;
}

template <int NCP, bool DUMP, int MODE, int TAB>
static cudaError_t launch_raw_pc_t(const RansLaunch &p, const DevArenas &a, cudaStream_t st) {
  auto k = rans_raw_pc_kernel<NCP, DUMP, MODE, TAB>;
  const PcGeom pc = dcb_pc_geom(p, 4u * NCP);
  const uint32_t pairs = std::max(1u, p.pairs);
  const uint32_t smem_bytes = pc.slice_bytes * pairs;
  if (smem_bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (e != cudaSuccess) return e;
  }
  cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  const uint32_t per_cta = p.lanes_per_warp * pairs;
  const uint32_t grid = (p.n_streams + per_cta - 1) / per_cta;
  k<<<grid, (p.split ? 128 : 64) * pairs, smem_bytes, st>>>(a.in, p.d_streams, p.d_order, p.n_streams, p.lanes_per_warp, pairs | (p.split ? 0x80000000u : 0u) | chain_low_bit(),
                                          pc_table_geom(p), pc, a.out, a.dbg, a.aux, p.dump | pc_no_split_bit());
  return cudaGetLastError();
}

cudaError_t dcb_launch_rans_raw_pc(const RansLaunch &p, int ncp, const DevArenas &a, cudaStream_t st) {
  if (!p.dump) {
#define DCB_SPEC(M, N)                                                                 \
  if (p.mode == M && ncp == N)                                                         \
    return p.compact ? launch_raw_pc_t<N, false, M, 2>(p, a, st) : launch_raw_pc_t<N, false, M, 1>(p, a, st);
    DCB_SPEC(1, 3)
    DCB_SPEC(1, 2)
    DCB_SPEC(2, 3)
    DCB_SPEC(2, 4)
    DCB_SPEC(3, 2)
    DCB_SPEC(4, 3)
    DCB_SPEC(4, 2)
#undef DCB_SPEC
  }
#define DCB_CASE(N) \
  case N:           \
    return p.dump ? launch_raw_pc_t<N, true, 0, 0>(p, a, st) : launch_raw_pc_t<N, false, 0, 0>(p, a, st);
  switch (ncp) {
    DCB_CASE(1)
    DCB_CASE(2)
    DCB_CASE(3)
    DCB_CASE(4)
    default:
      return cudaErrorInvalidValue;
  }
#undef DCB_CASE
}

cudaError_t dcb_launch_rans_tag_pc(const RansLaunch &p, const DevArenas &a, cudaStream_t st) {
  const PcGeom pc = dcb_pc_geom(p, 16u);
  const uint32_t pairs = std::max(1u, p.pairs);
  const uint32_t smem_bytes = pc.slice_bytes * pairs;
  if (smem_bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(rans_tag_pc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (e != cudaSuccess) return e;
  }
  cudaFuncSetAttribute(rans_tag_pc_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  const uint32_t per_cta = p.lanes_per_warp * pairs;
  const uint32_t grid = (p.n_streams + per_cta - 1) / per_cta;
  rans_tag_pc_kernel<<<grid, (p.split ? 128 : 64) * pairs, smem_bytes, st>>>(a.in, p.d_streams, p.d_order, p.n_streams, p.lanes_per_warp,
                                                            pairs | (p.split ? 0x80000000u : 0u) | chain_low_bit(), pc_table_geom(p), pc, a.aux);
  return cudaGetLastError();
}
