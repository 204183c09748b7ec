// draco_sharp_b200/csrc/dcb_faces.cu -- faces of meshes in the output arena (DCB_FACES_ARENA).
//
// Every mesh buffer's faces (3 u32 point ids per face, Mesh.Faces) land in a region of the output arena.  Two kernels fill
// the regions of a shard, each in one launch for all of its jobs (jobs found through running sums of their sizes):
//   seq_plain_kernel   one thread per 4 indices: fixed-width plain indices of sequential meshes (connectivity method 1,
//                      1, 2 or 4 bytes each, MeshSequentialDecoder.cs:58-77) widened to u32, and faces that are already
//                      u32 in the maps arena (Edgebreaker faces, host-decoded sequential faces) copied with 16-byte loads
//   seq_varint_kernel  one CTA per 4 KiB chunk of a varint index run (65536 <= points < 2^21): each thread marks the
//                      terminator bytes (bit 7 clear) of 16 bytes, a block scan from the chunk's checkpoint (indices that
//                      end in front of it, counted by the host while it located the run) gives every terminator its
//                      index, and the terminator's thread assembles the value backwards over the continuation bytes in
//                      front of it -- the low 32 bits of what DecoderBuffer's varint read gives (Reader::varint in
//                      dcb_mesh_host.cu).  The host has checked the framing (no varint longer than 10 bytes, no run
//                      leaving the buffer), so nothing here can fail.
//   seq_index_*        Raw index differences of sequential meshes (method 0, MeshSequentialDecoder.cs:86-110): the
//                      Raw rANS kernels decode them as one more one-component stream without zig-zag into the int32
//                      scratch; a two-pass chunk-sum scan turns the sign-magnitude steps into indices (sum pass: one CTA
//                      per 4096 indices, their sum and the extremes of their running prefix; base pass: one thread per
//                      buffer walks its chunk sums, checks every chunk's extremes against 0 and INT32_MAX and fails the
//                      buffer with DCB_ERR_CONNECTIVITY as dcb_host_sequential does; store pass: the chunks again).
// Product code: nothing here touches oracle/.
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>

#include "dcb_internal.h"
#include "dcb_jobs.cuh"
#include "dcb_kernels.h"

namespace {

constexpr uint32_t kThreads = 256;
constexpr uint32_t kPerThread = 4;
constexpr uint32_t kTile = kThreads * kPerThread;
constexpr uint32_t kVarintBytes = DCB_VARINT_CHUNK / kThreads;  // bytes of a chunk per thread
static_assert(kVarintBytes * kThreads == DCB_VARINT_CHUNK, "a varint chunk is one CTA iteration");

__global__ void __launch_bounds__(kThreads) seq_plain_kernel(FaceStage p, const uint8_t *__restrict__ in,
                                                             const uint8_t *__restrict__ maps, uint8_t *__restrict__ out) {
  dcb_for_each_element<kThreads, kPerThread>(p.unit_prefix, p.n_plain, [&](uint32_t j, uint64_t u) {
    const FaceJob &f = p.plain[j];
    const uint64_t i0 = u * 4;
    const uint32_t cnt = (uint32_t)(f.n_idx - i0 < 4 ? f.n_idx - i0 : 4);
    uint32_t v[4] = {0, 0, 0, 0};
    if (f.from_maps) {  // u32 faces on a 16-byte boundary of the maps arena
      const uint32_t *src = reinterpret_cast<const uint32_t *>(maps + f.src_off) + i0;
      if (cnt == 4) {
        const uint4 q = __ldg(reinterpret_cast<const uint4 *>(src));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
      } else {
        for (uint32_t k = 0; k < cnt; ++k) v[k] = __ldg(src + k);
      }
    } else {  // little-endian indices at any byte offset of the input arena
      const uint32_t w = f.width;
      const uint8_t *src = in + f.src_off + i0 * w;
      for (uint32_t k = 0; k < cnt; ++k)
        for (uint32_t b = 0; b < w; ++b) v[k] |= (uint32_t)__ldg(src + k * w + b) << (8 * b);
    }
    uint32_t *dst = reinterpret_cast<uint32_t *>(out + f.dst_off) + i0;
    if (cnt == 4) *reinterpret_cast<uint4 *>(dst) = make_uint4(v[0], v[1], v[2], v[3]);
    else
      for (uint32_t k = 0; k < cnt; ++k) dst[k] = v[k];
  });
}

// exclusive scan of x over the CTA (kThreads threads); every thread must call it
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T x, T *s_warp) {
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  T inc = x;
#pragma unroll
  for (uint32_t d = 1; d < 32; d <<= 1) {
    const T y = __shfl_up_sync(0xFFFFFFFFu, inc, d);
    if (lane >= d) inc += y;
  }
  if (lane == 31) s_warp[w] = inc;
  __syncthreads();
  if (w == 0) {
    constexpr uint32_t kWarps = kThreads / 32;
    T s = lane < kWarps ? s_warp[lane] : T(0);
#pragma unroll
    for (uint32_t d = 1; d < kWarps; d <<= 1) {
      const T y = __shfl_up_sync(0xFFFFFFFFu, s, d);
      if (lane >= d) s += y;
    }
    if (lane < kWarps) s_warp[lane] = s;
  }
  __syncthreads();
  const T r = inc - x + (w ? s_warp[w - 1] : T(0));
  __syncthreads();  // s_warp is reused by the next call
  return r;
}

__global__ void __launch_bounds__(kThreads) seq_varint_kernel(FaceStage p, const uint8_t *__restrict__ in, uint8_t *__restrict__ out) {
  __shared__ uint32_t s_warp[kThreads / 32];
  for (uint64_t c = blockIdx.x; c < p.total_chunks; c += gridDim.x) {
    const uint32_t j = dcb_find_job(p.chunk_prefix, p.n_varint, c);
    const FaceJob &f = p.varint[j];
    const uint64_t lc = c - p.chunk_prefix[j];
    const uint8_t *run = in + f.src_off;
    const uint64_t b0 = lc * DCB_VARINT_CHUNK + (uint64_t)threadIdx.x * kVarintBytes;
    const uint32_t nb = (uint32_t)(b0 >= f.n_bytes ? 0 : (f.n_bytes - b0 < kVarintBytes ? f.n_bytes - b0 : kVarintBytes));
    uint32_t ends = 0;  // bit k: byte b0 + k ends a varint
    for (uint32_t k = 0; k < nb; ++k)
      if (!(__ldg(run + b0 + k) & 0x80u)) ends |= 1u << k;
    uint64_t ord = __ldg(p.ckpt + f.ckpt_off + lc) + block_exclusive_scan<uint32_t>((uint32_t)__popc(ends), s_warp);
    uint32_t *dst = reinterpret_cast<uint32_t *>(out + f.dst_off);
    while (ends) {
      const uint32_t k = (uint32_t)__ffs(ends) - 1u;
      ends &= ends - 1u;
      uint64_t q = b0 + k;
      uint32_t v = __ldg(run + q) & 0x7Fu;
      while (q > 0) {  // continuation bytes in front of the terminator, back to the previous terminator or the run start
        const uint32_t byte = __ldg(run + q - 1);
        if (!(byte & 0x80u)) break;
        v = (v << 7) | (byte & 0x7Fu);
        --q;
      }
      dst[ord++] = v;
    }
  }
}

constexpr uint32_t kIndexPerThread = DCB_INDEX_CHUNK / kThreads;
static_assert(kIndexPerThread * kThreads == DCB_INDEX_CHUNK, "an index chunk is one CTA iteration");

// sign-magnitude step of one index symbol (the bitstream's rule; dcb_host_sequential)
__device__ __forceinline__ int64_t index_step(int32_t sym) {
  const int64_t m = (int64_t)((uint32_t)sym >> 1);
  return (sym & 1) ? -m : m;
}

// the chunk c of the index jobs: its job, the job's symbols and the chunk's first index inside the job
struct IndexChunk {
  uint32_t j;
  uint64_t i0, n;  // first index of the chunk, indices in it
};
__device__ __forceinline__ IndexChunk index_chunk(const FaceStage &p, uint64_t c) {
  IndexChunk k;
  k.j = dcb_find_job(p.index_prefix, p.n_index, c);
  k.i0 = (c - p.index_prefix[k.j]) * DCB_INDEX_CHUNK;
  const uint64_t n_idx = p.index[k.j].n_idx;
  k.n = n_idx - k.i0 < DCB_INDEX_CHUNK ? n_idx - k.i0 : DCB_INDEX_CHUNK;
  return k;
}

// the running prefix of a thread's kIndexPerThread steps, relative to the chunk start (exclusive scan over the CTA)
__device__ __forceinline__ void chunk_prefixes(const int32_t *sym, uint64_t n, int64_t *s_warp, int64_t (&pre)[kIndexPerThread],
                                               int64_t &excl) {
  const uint64_t t0 = (uint64_t)threadIdx.x * kIndexPerThread;
  int64_t acc = 0;
#pragma unroll
  for (uint32_t k = 0; k < kIndexPerThread; ++k) {
    if (t0 + k < n) acc += index_step(__ldg(sym + t0 + k));
    pre[k] = acc;
  }
  excl = block_exclusive_scan<int64_t>(acc, s_warp);
}

__global__ void __launch_bounds__(kThreads) seq_index_sum_kernel(FaceStage p, const uint8_t *__restrict__ aux,
                                                                 const StreamDesc *__restrict__ streams) {
  __shared__ int64_t s_warp[kThreads / 32];
  __shared__ int64_t s_min[kThreads / 32], s_max[kThreads / 32];
  for (uint64_t c = blockIdx.x; c < p.total_index_chunks; c += gridDim.x) {
    const IndexChunk k = index_chunk(p, c);
    const FaceJob &f = p.index[k.j];
    const int32_t *sym = reinterpret_cast<const int32_t *>(aux + streams[f.stream].aux_off) + k.i0;
    int64_t pre[kIndexPerThread], excl;
    chunk_prefixes(sym, k.n, s_warp, pre, excl);
    const uint64_t t0 = (uint64_t)threadIdx.x * kIndexPerThread;
    int64_t mn = INT64_MAX, mx = INT64_MIN;
#pragma unroll
    for (uint32_t q = 0; q < kIndexPerThread; ++q)
      if (t0 + q < k.n) {
        mn = min(mn, excl + pre[q]);
        mx = max(mx, excl + pre[q]);
      }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = min(mn, (int64_t)__shfl_xor_sync(0xFFFFFFFFu, mn, o));
      mx = max(mx, (int64_t)__shfl_xor_sync(0xFFFFFFFFu, mx, o));
    }
    if ((threadIdx.x & 31u) == 0) {
      s_min[threadIdx.x >> 5] = mn;
      s_max[threadIdx.x >> 5] = mx;
    }
    __syncthreads();
    if (threadIdx.x == kThreads - 1) {  // the last thread's inclusive prefix is the chunk's sum
      int64_t cmn = s_min[0], cmx = s_max[0];
      for (uint32_t w = 1; w < kThreads / 32; ++w) {
        cmn = min(cmn, s_min[w]);
        cmx = max(cmx, s_max[w]);
      }
      p.chunk_sum[c] = excl + pre[kIndexPerThread - 1];
      p.chunk_min[c] = cmn;
      p.chunk_max[c] = cmx;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kThreads) seq_index_base_kernel(FaceStage p, const StreamDesc *__restrict__ streams) {
  for (uint32_t j = blockIdx.x * kThreads + threadIdx.x; j < p.n_index; j += gridDim.x * kThreads) {
    int32_t st = streams[p.index[j].stream].status;  // the rANS stream failed: its status is the buffer's
    int64_t base = 0;
    for (uint64_t c = p.index_prefix[j]; c < p.index_prefix[j + 1]; ++c) {
      if (!st && (base + p.chunk_min[c] < 0 || base + p.chunk_max[c] > 0x7FFFFFFFll)) st = DCB_ERR_CONNECTIVITY;
      const int64_t s = p.chunk_sum[c];
      p.chunk_sum[c] = base;
      base += s;
    }
    p.status[j] = st;
  }
}

__global__ void __launch_bounds__(kThreads) seq_index_store_kernel(FaceStage p, const uint8_t *__restrict__ aux,
                                                                   const StreamDesc *__restrict__ streams, uint8_t *__restrict__ out) {
  __shared__ int64_t s_warp[kThreads / 32];
  for (uint64_t c = blockIdx.x; c < p.total_index_chunks; c += gridDim.x) {
    const IndexChunk k = index_chunk(p, c);
    if (p.status[k.j]) continue;  // uniform over the CTA
    const FaceJob &f = p.index[k.j];
    const int32_t *sym = reinterpret_cast<const int32_t *>(aux + streams[f.stream].aux_off) + k.i0;
    int64_t pre[kIndexPerThread], excl;
    chunk_prefixes(sym, k.n, s_warp, pre, excl);
    const int64_t base = p.chunk_sum[c] + excl;
    uint32_t *dst = reinterpret_cast<uint32_t *>(out + f.dst_off) + k.i0;
    const uint64_t t0 = (uint64_t)threadIdx.x * kIndexPerThread;
#pragma unroll
    for (uint32_t q = 0; q < kIndexPerThread; q += 4) {
      if (t0 + q + 4 <= k.n) {
        *reinterpret_cast<uint4 *>(dst + t0 + q) = make_uint4((uint32_t)(base + pre[q]), (uint32_t)(base + pre[q + 1]),
                                                              (uint32_t)(base + pre[q + 2]), (uint32_t)(base + pre[q + 3]));
      } else {
        for (uint32_t r = q; r < kIndexPerThread && t0 + r < k.n; ++r) dst[t0 + r] = (uint32_t)(base + pre[r]);
      }
    }
  }
}

uint32_t grid_for(uint64_t units, uint32_t num_sms) {
  return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(units, (uint64_t)num_sms * 8));
}

}  // namespace

cudaError_t dcb_launch_faces(const FaceStage &p, const StreamDesc *d_streams, const DevArenas &a, uint32_t num_sms, cudaStream_t st) {
  if (p.n_index) {
    if (p.total_index_chunks) seq_index_sum_kernel<<<grid_for(p.total_index_chunks, num_sms), kThreads, 0, st>>>(p, a.aux, d_streams);
    seq_index_base_kernel<<<grid_for((p.n_index + kThreads - 1) / kThreads, num_sms), kThreads, 0, st>>>(p, d_streams);
    if (p.total_index_chunks)
      seq_index_store_kernel<<<grid_for(p.total_index_chunks, num_sms), kThreads, 0, st>>>(p, a.aux, d_streams, a.out);
  }
  if (p.total_units)
    seq_plain_kernel<<<grid_for((p.total_units + kTile - 1) / kTile, num_sms), kThreads, 0, st>>>(p, a.in, a.maps, a.out);
  if (p.total_chunks) seq_varint_kernel<<<grid_for(p.total_chunks, num_sms), kThreads, 0, st>>>(p, a.in, a.out);
  return cudaGetLastError();
}
