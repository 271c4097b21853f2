// doc_filter.cu — edits of the document bitmaps that the filtered K2 / K4 entry points read (include/lr_b200.h).
//
// Deleting or restoring a document is a bit flip in the `live` bitmap, enqueued on the stream that runs the searches:
// no host synchronisation, no allocation, so a serving process can issue it between CUDA-graph replays (or capture it).
#include "common.cuh"

namespace lr {

__global__ void doc_bitmap_update_kernel(uint32_t* __restrict__ words, int64_t ld_words, const int64_t* __restrict__ ids,
                                         int64_t n, int set) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t id = ids[i];
    if (id < 0 || id >= ld_words * 32) continue;  // ids outside the bitmap are ignored
    const uint32_t bit = 1u << (id & 31);
    if (set) atomicOr(words + (id >> 5), bit);
    else atomicAnd(words + (id >> 5), ~bit);
  }
}

}  // namespace lr

using namespace lr;

extern "C" int lr_doc_bitmap_update(uint32_t* words, int64_t ld_words, const int64_t* ids, int64_t n, int set,
                                    void* stream) {
  LR_CHECK_ARG(words && ld_words >= 1, "doc_bitmap_update: null words or ld_words (%lld) < 1", (long long)ld_words);
  LR_CHECK_ARG(n >= 0 && (ids || n == 0), "doc_bitmap_update: null ids or n (%lld) < 0", (long long)n);
  LR_CHECK_ARG(set == 0 || set == 1, "doc_bitmap_update: set (%d) must be 0 or 1", set);
  if (n == 0) return LR_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  doc_bitmap_update_kernel<<<unsigned(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(words, ld_words, ids, n, set);
  LR_LAUNCH_CHECK();
  return LR_OK;
}
