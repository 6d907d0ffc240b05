// block_copy.cuh — the per-CTA byte copy / clear shared by k_masked_bytes (episode_kernel.cu) and k_snapshot
// (snapshot_kernel.cu): one CTA moves one contiguous slice.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace ag {

// d[0, n) = s[0, n) (kCopy) or zeros, by all threads of the CTA.  d and s must share their alignment modulo 16: both
// then have the same head in front of the first 16-byte boundary; the body moves in 16-byte vectors, four in flight per
// thread, and the tail byte by byte.
template <bool kCopy>
__device__ __forceinline__ void block_copy(uint8_t* __restrict__ d, const uint8_t* __restrict__ s, size_t n) {
  size_t head = (16u - ((uintptr_t)d & 15u)) & 15u;
  if (head > n) head = n;
  const size_t nvec = (n - head) / 16, tail = head + nvec * 16;
  const int t = threadIdx.x, nt = blockDim.x;
  for (size_t k = t; k < head; k += nt) d[k] = kCopy ? s[k] : 0;
  for (size_t k = tail + t; k < n; k += nt) d[k] = kCopy ? s[k] : 0;
  uint4* dv = reinterpret_cast<uint4*>(d + head);
  const uint4* sv = kCopy ? reinterpret_cast<const uint4*>(s + head) : nullptr;
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  size_t k = t;
  for (; k + 3 * (size_t)nt < nvec; k += 4 * (size_t)nt) {
    uint4 v0 = z, v1 = z, v2 = z, v3 = z;
    if (kCopy) { v0 = sv[k]; v1 = sv[k + nt]; v2 = sv[k + 2 * nt]; v3 = sv[k + 3 * nt]; }
    dv[k] = v0; dv[k + nt] = v1; dv[k + 2 * nt] = v2; dv[k + 3 * nt] = v3;
  }
  for (; k < nvec; k += nt) dv[k] = kCopy ? sv[k] : z;
}

}  // namespace ag
