// draco_sharp_b200/csrc/dcb_jobs.cuh -- element-parallel loops over a list of jobs of different sizes, the jobs found
// through running sums of their sizes (point stage, dcb_points.cu; faces stage, dcb_faces.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// last job j with prefix[j] <= i (prefix: n + 1 non-decreasing running sums, i < prefix[n])
__device__ __forceinline__ uint32_t dcb_find_job(const uint64_t *prefix, uint32_t n, uint64_t i) {
  uint32_t lo = 0, hi = n;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (prefix[mid] <= i) lo = mid;
    else hi = mid;
  }
  return lo;
}

// f(job, index inside the job) over the elements [0, prefix[n]) of n jobs, Threads * PerThread consecutive elements per
// block iteration: one binary search per tile, then every thread walks forward (jobs are contiguous, elements of a
// thread increase)
template <uint32_t Threads, uint32_t PerThread, typename F>
__device__ __forceinline__ void dcb_for_each_element(const uint64_t *prefix, uint32_t n, F &&f) {
  constexpr uint32_t kTile = Threads * PerThread;
  __shared__ uint32_t s_job;
  const uint64_t total = prefix[n];
  for (uint64_t t0 = (uint64_t)blockIdx.x * kTile; t0 < total; t0 += (uint64_t)gridDim.x * kTile) {
    __syncthreads();
    if (threadIdx.x == 0) s_job = dcb_find_job(prefix, n, t0);
    __syncthreads();
    uint32_t j = s_job;
    uint64_t next = prefix[j + 1];
#pragma unroll
    for (uint32_t k = 0; k < PerThread; ++k) {
      const uint64_t i = t0 + k * Threads + threadIdx.x;
      if (i >= total) break;
      while (i >= next) next = prefix[++j + 1];
      f(j, i - prefix[j]);
    }
  }
}
