// warp_topk.cuh — exact per-warp cut of a candidate list to its top-k (K4 and the forward-segment kernel).
#pragma once
#include "common.cuh"

namespace lr {

// Exact cut of list[0..n) (n > k) to its k largest keys, in place; returns the new threshold key (every kept key is
// >= it, every dropped key < it).  One warp; hist = 256 words of this warp's shared memory.  Out of line: it runs a few
// times per unit and must not bloat the step loop's instruction footprint.
inline __device__ __noinline__ uint64_t warp_cut_topk(uint64_t* list, uint32_t* n_io, int k, uint32_t* hist) {
  const uint32_t full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const uint32_t n = *n_io;
  uint64_t prefix = 0, kstar = 0;
  uint32_t remaining = uint32_t(k);
  for (int pass = 7; pass >= 0; --pass) {
    const int shift = pass * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) hist[lane + 32 * i] = 0;
    __syncwarp();
    for (uint32_t i = lane; i < n; i += 32) {
      const uint64_t key = list[i];
      if (pass == 7 || (key >> (shift + 8)) == prefix) atomicAdd(&hist[(key >> shift) & 0xFFu], 1u);
    }
    __syncwarp();
    uint32_t bin, rem2;
    bool take_all;
    warp_find_bin_desc(hist, remaining, bin, rem2, take_all);
    __syncwarp();
    prefix = (prefix << 8) | uint64_t(bin);
    remaining = rem2;
    if (take_all || pass == 0) {
      kstar = prefix << shift;
      break;
    }
  }
  uint32_t m = 0;
  for (uint32_t i0 = 0; i0 < n; i0 += 32) {
    const uint32_t i = i0 + lane;
    const uint64_t key = i < n ? list[i] : 0ull;
    const bool keep = i < n && key >= kstar;
    const uint32_t km = __ballot_sync(full, keep);
    __syncwarp();
    if (keep) list[m + __popc(km & lanemask_lt())] = key;
    m += __popc(km);
    __syncwarp();
  }
  *n_io = m;
  return kstar;
}

}  // namespace lr
