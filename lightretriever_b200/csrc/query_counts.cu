// query_counts.cu — the sparse query of the online path: token counts per bag, on device.
//
// Replaces the host parse of the pseudo-query  Counter(ids)  (reference inference/exact_search_base.py:371-435,
// sparse_search.parse_queries here) and its "bow" form  {t: 1 for t in set(ids)}  (exact_search_base.py:398-424),
// for the query token ids the notebook hands to the sparse searcher (scripts/asymmetric_sparse_infer.ipynb:50).
//
// Two launches, no host synchronisation, nothing allocated: safe inside CUDA-graph capture.
//   1. one CTA per bag: the bag's in-range ids are gathered into shared memory as int32 keys (an id outside [0, V) is
//      dropped), padded to a power of two with a sentinel that sorts last, bitonic-sorted, and every run of equal keys
//      becomes one (token, count) term.  The bag's terms go to the scratch rows [beg, beg + terms) of the bag's own id
//      range, their number to scratch counts[b].
//   2. one CTA: exclusive scan of the per-bag term counts -> q_indptr, then every bag's terms are copied to their place
//      in q_tok / q_cnt, and the tail [q_indptr[n_bags], n_ids) is zeroed so that the whole output is deterministic.
#include "common.cuh"

namespace lr {

constexpr int QC_THREADS = 256;
constexpr int QC_SCAN_THREADS = 1024;
constexpr int32_t QC_SENTINEL = 0x7FFFFFFF;  // > every valid id (V <= 2^31 - 1)

static size_t qc_align(size_t b) { return (b + 255) & ~size_t(255); }

// Block-wide exclusive scan of one int per thread; returns the prefix, *total = the sum over the block.
template <int THREADS>
__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_sums, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int y = __shfl_up_sync(0xFFFFFFFFu, x, off);
    if (lane >= off) x += y;
  }
  if (lane == 31) warp_sums[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = lane < THREADS / 32 ? warp_sums[lane] : 0;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int y = __shfl_up_sync(0xFFFFFFFFu, w, off);
      if (lane >= off) w += y;
    }
    if (lane < THREADS / 32) warp_sums[lane] = w;  // inclusive
  }
  __syncthreads();
  const int base = warp ? warp_sums[warp - 1] : 0;
  *total = warp_sums[THREADS / 32 - 1];
  __syncthreads();  // warp_sums may be reused by the caller's next scan
  return base + x - v;
}

// dynamic smem: int32 keys[cap] + int32 head positions[cap + 1], cap = the power of two >= max_bag
__global__ void __launch_bounds__(QC_THREADS)
query_counts_bag_kernel(const int64_t* __restrict__ ids, const int64_t* __restrict__ offsets, int64_t n_ids,
                        int64_t n_bags, int64_t V, int64_t max_bag, int bow, int32_t* __restrict__ s_tok,
                        int32_t* __restrict__ s_cnt, int32_t* __restrict__ s_terms, int32_t* err_flag) {
  extern __shared__ int32_t qc_smem[];
  __shared__ int warp_sums[QC_THREADS / 32];
  __shared__ int s_valid;
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x;
  const int64_t beg = offsets[b];
  const int64_t end = (b + 1 < n_bags) ? offsets[b + 1] : n_ids;
  int32_t* key = qc_smem;
  if (tid == 0) s_valid = 0;
  __syncthreads();
  // a bag outside [0, n_ids], or one that ends before it starts (descending offsets would let bags overlap), flags the
  // call and stays empty
  const bool bad_range = beg < 0 || end < beg || end > n_ids;
  if (!bad_range) {
    // in-range ids are gathered in any order (they are sorted next); an id outside [0, V) -- the searcher's -1 padding
    // included -- contributes nothing and takes no slot
    for (int64_t i = beg + tid; i < end; i += QC_THREADS) {
      const int64_t id = ids[i];
      if (id >= 0 && id < V) {
        const int pos = atomicAdd(&s_valid, 1);
        if (pos < max_bag) key[pos] = int32_t(id);
      }
    }
  }
  __syncthreads();
  const int n_valid = s_valid;
  if (bad_range || n_valid > max_bag) {  // more in-range ids than the host's bound: flagged, empty
    if (tid == 0) {
      s_terms[b] = 0;
      if (err_flag) atomicOr(err_flag, 1);
    }
    return;
  }
  int npad = 1;
  while (npad < n_valid) npad <<= 1;
  int32_t* head = qc_smem + npad;
  for (int i = n_valid + tid; i < npad; i += QC_THREADS) key[i] = QC_SENTINEL;
  __syncthreads();
  // bitonic sort, ascending
  for (int size = 2; size <= npad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < npad / 2; t += QC_THREADS) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const int32_t a = key[lo], c = key[hi];
        if (((lo & size) == 0) == (a > c)) {
          key[lo] = c;
          key[hi] = a;
        }
      }
      __syncthreads();
    }
  }
  // run heads: every thread owns a contiguous piece of `per` slots, so ranks follow the sorted order
  const int per = (npad + QC_THREADS - 1) / QC_THREADS;
  const int i0 = tid * per, i1 = min(i0 + per, npad);
  int mine = 0;
  for (int i = i0; i < i1; ++i) mine += key[i] != QC_SENTINEL && (i == 0 || key[i - 1] != key[i]);
  int terms;
  int r = block_exclusive_scan<QC_THREADS>(mine, warp_sums, &terms);
  for (int i = i0; i < i1; ++i) {
    const int32_t k = key[i];
    if (k == QC_SENTINEL) {
      if (i == 0 || key[i - 1] != QC_SENTINEL) head[terms] = i;  // first sentinel = end of the last run
      continue;
    }
    if (i == 0 || key[i - 1] != k) head[r++] = i;
  }
  if (tid == 0 && key[npad - 1] != QC_SENTINEL) head[terms] = npad;  // no sentinel at all
  __syncthreads();
  for (int j = tid; j < terms; j += QC_THREADS) {
    const int p = head[j];
    s_tok[beg + j] = key[p];
    s_cnt[beg + j] = bow ? 1 : head[j + 1] - p;
  }
  if (tid == 0) s_terms[b] = terms;
}

__global__ void __launch_bounds__(QC_SCAN_THREADS)
query_counts_compact_kernel(const int64_t* __restrict__ offsets, int64_t n_ids, int64_t n_bags,
                            const int32_t* __restrict__ s_tok, const int32_t* __restrict__ s_cnt,
                            const int32_t* __restrict__ s_terms, int32_t* __restrict__ q_indptr,
                            int32_t* __restrict__ q_tok, int32_t* __restrict__ q_cnt, int32_t* err_flag) {
  __shared__ int warp_sums[QC_SCAN_THREADS / 32];
  const int tid = threadIdx.x;
  int64_t carry = 0;
  for (int64_t c0 = 0; c0 < n_bags; c0 += QC_SCAN_THREADS) {
    const int64_t b = c0 + tid;
    const int v = b < n_bags ? s_terms[b] : 0;
    int chunk;
    const int ex = block_exclusive_scan<QC_SCAN_THREADS>(v, warp_sums, &chunk);
    if (b < n_bags) q_indptr[b] = int32_t(carry + ex);
    carry += chunk;
  }
  // bags that overlap (offsets not ascending) could hold more terms than the output has rows: flag, return all empty
  const bool overflow = carry > n_ids;
  if (tid == 0) q_indptr[n_bags] = overflow ? 0 : int32_t(carry);
  if (overflow) {
    for (int64_t b = tid; b < n_bags; b += QC_SCAN_THREADS) q_indptr[b] = 0;
    for (int64_t i = tid; i < n_ids; i += QC_SCAN_THREADS) q_tok[i] = q_cnt[i] = 0;
    if (tid == 0 && err_flag) atomicOr(err_flag, 1);
    return;
  }
  __syncthreads();  // q_indptr written above is read back by other threads of this CTA
  const int lane = tid & 31, warp = tid >> 5;
  for (int64_t b = warp; b < n_bags; b += QC_SCAN_THREADS / 32) {
    const int64_t src = offsets[b];
    const int n = s_terms[b];
    const int64_t dst = q_indptr[b];
    for (int j = lane; j < n; j += 32) {
      q_tok[dst + j] = s_tok[src + j];
      q_cnt[dst + j] = s_cnt[src + j];
    }
  }
  for (int64_t i = carry + tid; i < n_ids; i += QC_SCAN_THREADS) q_tok[i] = q_cnt[i] = 0;
}

}  // namespace lr

using namespace lr;

extern "C" size_t lr_query_token_counts_scratch_bytes(int64_t n_ids, int64_t n_bags) {
  if (n_ids < 0 || n_bags < 1) return 0;
  const size_t rows = size_t(n_ids > 0 ? n_ids : 1);
  return 2 * qc_align(rows * 4) + qc_align(size_t(n_bags) * 4);
}

extern "C" int lr_query_token_counts(const int64_t* ids, const int64_t* offsets, int64_t n_ids, int64_t n_bags, int64_t V,
                                     int64_t max_bag, int bow, int32_t* q_indptr, int32_t* q_tok, int32_t* q_cnt,
                                     int32_t* err_flag, void* scratch, size_t scratch_bytes, void* stream) {
  LR_CHECK_ARG(n_bags >= 1 && n_ids >= 0, "query_token_counts: need n_bags >= 1 and n_ids >= 0");
  LR_CHECK_ARG(offsets && q_indptr && scratch, "query_token_counts: null pointer");
  LR_CHECK_ARG(n_ids == 0 || (ids && q_tok && q_cnt), "query_token_counts: null ids / q_tok / q_cnt");
  LR_CHECK_ARG(n_ids < (int64_t(1) << 31) && n_bags < (int64_t(1) << 31), "query_token_counts: too many ids or bags");
  LR_CHECK_ARG(V >= 1 && V <= int64_t(QC_SENTINEL), "query_token_counts: V (%lld) must be in [1, 2^31 - 1]", (long long)V);
  LR_CHECK_ARG(max_bag >= 0 && max_bag <= LR_QUERY_MAX_BAG, "query_token_counts: max_bag (%lld) must be in [0, %d]",
               (long long)max_bag, LR_QUERY_MAX_BAG);
  LR_CHECK_ARG(bow == 0 || bow == 1, "query_token_counts: bow must be 0 or 1");
  const size_t need = lr_query_token_counts_scratch_bytes(n_ids, n_bags);
  if (scratch_bytes < need) {
    set_error("query_token_counts: scratch of %zu bytes, need %zu", scratch_bytes, need);
    return LR_EWORKSPACE;
  }
  const size_t rows = qc_align(size_t(n_ids > 0 ? n_ids : 1) * 4);
  int32_t* s_tok = static_cast<int32_t*>(scratch);
  int32_t* s_cnt = reinterpret_cast<int32_t*>(static_cast<char*>(scratch) + rows);
  int32_t* s_terms = reinterpret_cast<int32_t*>(static_cast<char*>(scratch) + 2 * rows);
  int npad = 1;
  while (npad < max_bag) npad <<= 1;
  const int smem = (2 * npad + 1) * 4;
  int rc = ensure_dyn_smem(reinterpret_cast<const void*>(query_counts_bag_kernel), (2 * LR_QUERY_MAX_BAG + 1) * 4);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  query_counts_bag_kernel<<<unsigned(n_bags), QC_THREADS, smem, st>>>(ids, offsets, n_ids, n_bags, V, max_bag, bow,
                                                                       s_tok, s_cnt, s_terms, err_flag);
  LR_LAUNCH_CHECK();
  query_counts_compact_kernel<<<1, QC_SCAN_THREADS, 0, st>>>(offsets, n_ids, n_bags, s_tok, s_cnt, s_terms, q_indptr,
                                                             q_tok, q_cnt, err_flag);
  LR_LAUNCH_CHECK();
  return LR_OK;
}
