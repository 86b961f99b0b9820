// Device exclusive scan of int counts (DESIGN 7c: count -> three-kernel exclusive scan -> fill), shared by the snap grid
// (snap.cu) and the OBJ parser (obj_parse.cu).
//
// Layout the caller guarantees: `counts` holds n_pad ints, n_pad a multiple of kScanItems and at most
// kScanItems * kScanMaxBlocks, 16-byte aligned, padding zero; `block_sums` holds kScanMaxBlocks ints.
#pragma once

#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "common.cuh"

namespace mvlm {

constexpr int kScanItems = 4096;      // counts per scan block (256 threads x 16)
constexpr int kScanMaxBlocks = 4096;  // one 1024-thread block scans the block sums (4 each)

namespace {

__global__ void __launch_bounds__(256) scan_a_kernel(const int* __restrict__ counts, int* __restrict__ block_sums) {
  using Reduce = cub::BlockReduce<int, 256>;
  __shared__ typename Reduce::TempStorage tmp;
  const int4* src = reinterpret_cast<const int4*>(counts + static_cast<size_t>(blockIdx.x) * kScanItems) + threadIdx.x * 4;
  int sum = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int4 v = src[i];
    sum += v.x + v.y + v.z + v.w;
  }
  const int total = Reduce(tmp).Sum(sum);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) scan_b_kernel(int* __restrict__ block_sums, int nb, int* __restrict__ total_out) {
  using Scan = cub::BlockScan<int, 1024>;
  __shared__ typename Scan::TempStorage tmp;
  int v[4], sum = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int j = threadIdx.x * 4 + i;
    v[i] = j < nb ? block_sums[j] : 0;
    sum += v[i];
  }
  int excl, total;
  Scan(tmp).ExclusiveSum(sum, excl, total);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int j = threadIdx.x * 4 + i;
    if (j < nb) block_sums[j] = excl;
    excl += v[i];
  }
  if (threadIdx.x == 0) *total_out = total;
}

__global__ void __launch_bounds__(256) scan_c_kernel(const int* __restrict__ counts, const int* __restrict__ block_sums,
                                                     int* __restrict__ out) {
  using Scan = cub::BlockScan<int, 256>;
  __shared__ typename Scan::TempStorage tmp;
  const size_t base = static_cast<size_t>(blockIdx.x) * kScanItems + threadIdx.x * 16;
  int v[16], sum = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int4 q = reinterpret_cast<const int4*>(counts + base)[i];
    v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
    sum += q.x + q.y + q.z + q.w;
  }
  int excl;
  Scan(tmp).ExclusiveSum(sum, excl);
  excl += block_sums[blockIdx.x];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int4 q;
    q.x = excl; excl += v[4 * i];
    q.y = excl; excl += v[4 * i + 1];
    q.z = excl; excl += v[4 * i + 2];
    q.w = excl; excl += v[4 * i + 3];
    reinterpret_cast<int4*>(out + base)[i] = q;
  }
}

// out[i] = counts[0] + ... + counts[i - 1] for i < n_pad, *total_out = the sum of all counts (device pointer).
// Three launches on s (counted by the caller).
inline void exclusive_scan(const int* counts, int n_pad, int* block_sums, int* out, int* total_out, cudaStream_t s) {
  const int nb = n_pad / kScanItems;
  scan_a_kernel<<<nb, 256, 0, s>>>(counts, block_sums);
  scan_b_kernel<<<1, 1024, 0, s>>>(block_sums, nb, total_out);
  scan_c_kernel<<<nb, 256, 0, s>>>(counts, block_sums, out);
}

}  // namespace
}  // namespace mvlm
