// sparse_score.cu — K4: sparse impact scoring + exact top-k over an inverted index.
//
// Replaces the Anserini / Lucene impact search of AnseriniSearch.retrieve_with_emb
// (reference retriever/anserini_search.py:143-216; io.anserini:anserini:0.25.0 SearchCollection -impact
// -pretokenized).  Score definition: scripts/asymmetric_sparse_infer.ipynb:207-228
//     score(q, d) = sum_{t in q ∩ d} count_q(t) * impact_d(t)        (integer arithmetic)
//
// Two kernels, chosen per batch ON THE DEVICE from the batch's mean posting run (sparse_density_kernel; both are launched
// and the one whose regime it is not returns at once):
//   * row kernel (sparse_rows.cuh) for DENSE batches — long posting runs, the Zipf head: rows of 32 postings of one
//     term, plain read-modify-write on warp-private accumulators, no shared-memory atomics;
//   * flat kernel (below, the round-1 design) for SPARSE batches — runs much shorter than a row.
// Common structure: gather-accumulate with warp-granular workers.  Documents are processed in blocks of SS_BLOCK_DOCS
// consecutive ids; every WARP is an independent worker with its own accumulator block, candidate list and histogram in
// shared memory, so neither kernel has a block-wide barrier and the dependent chain of one step (block pointers ->
// postings -> accumulators -> candidates) is hidden by the other resident warps.  A unit = (query, range of document
// blocks), handed out dynamically (one global atomic per unit).  Flat kernel, per step:
//   1. lane t owns query term t and walks its row of blockptr with a two-block-ahead prefetch: the posting
//      sub-range [blockptr[t][b], blockptr[t][b+1]) costs no search and no exposed latency;
//   2. the sub-ranges are flattened (warp scan + shuffle binary search) and streamed in batches of NB x 32 postings:
//      all loads of a batch are issued before its shared-memory atomicAdds;
//   3. the first add that finds 0 records the slot, so only touched accumulators are visited (a step touching more
//      than SS_TOUCH_CAP slots scans the block); entries beating the unit's running 64-bit threshold key — and the
//      query's global score floor, raised with atomicMax by every unit of that query — are appended to the warp's
//      candidate list; a full list is cut to its exact top-k by a warp-level 64-bit radix select.
// The unit's list goes to the workspace and the (two-level, for few queries) merge of topk_merge.cu produces the sorted
// result.  Integer-exact; 16-bit accumulators with a 32-bit second pass when a sum would overflow.
#include "common.cuh"
#include "warp_topk.cuh"

namespace lr {

int topk_merge_two_level(const uint64_t* keys, const int32_t* counts, int L, int64_t Q, int64_t q_stride, int cap, int k,
                         int score_kind, int64_t id_offset, float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                         int64_t out_key_stride, void* scratch, size_t scratch_bytes, cudaStream_t st);
size_t topk_merge_scratch_bytes(int L, int64_t Q, int cap, int k);

constexpr int SS_TOUCH_CAP = 512;  // touched-accumulator list per warp; a step that touches more scans the block
constexpr int SS_MAX_WARPS = 20;
constexpr int SS_BLOCK_DOCS = 4096;  // documents per index block = per accumulator block of the flat kernel
constexpr int SS_NB = 8;             // flat kernel: postings per lane in flight
constexpr int SS_DENSE_RUN = 24;     // mean postings per (query term, row-kernel step) from which a batch is dense

struct SSParams {
  const int32_t* q_indptr;
  const int32_t* q_tok;
  const int32_t* q_cnt;
  int64_t Q;
  const int64_t* post_indptr;
  const int32_t* post_doc;
  const uint16_t* post_imp;
  const uint32_t* blockptr;
  int64_t V, N;
  int nblk, S, k, cap, warp_bytes;
  int bd;             // documents per index block (blockptr granularity)
  uint64_t* unit_thr;  // row kernel: [S][Q] final threshold key of each finished unit (0 = not finished), zeroed per launch
  uint64_t* cand;     // [S][Q][cap]
  int32_t* counts;    // [S][Q]
  uint32_t* floor_q;  // [Q] score floor of each query (k-th best score some unit has proven), zeroed per launch
  uint32_t* next_unit;  // dynamic unit counter, zeroed per launch
  uint32_t* overflow;   // set by the 16-bit pass when an accumulator would exceed 65535; the 32-bit pass runs only then
  // regime dispatch: [0..1] = postings of all query terms of the batch (u64), [2] = number of query terms.  The batch is
  // DENSE when the mean posting run per (term, step of the row kernel) reaches dense_thresh; a kernel whose `want_dense`
  // disagrees returns at once.  Null: always run.
  const uint32_t* regime;
  uint32_t dense_thresh;
  int want_dense;
  DocFilter filter;  // documents a query may return (filter.on == 0: all); tested before a document is listed
};

__device__ __forceinline__ bool ss_regime_skip(const SSParams& p) {
  if (!p.regime) return false;
  const uint64_t postings = (uint64_t(p.regime[1]) << 32) | uint64_t(p.regime[0]);
  const bool dense = postings >= uint64_t(p.dense_thresh) * uint64_t(p.regime[2]);
  return dense != (p.want_dense != 0);
}

// Accumulator access.  AccT = uint16_t packs two documents per shared-memory word (twice the resident warps for the same
// block size); a sum that would not fit raises `ovf` and the launch is repeated with int32 accumulators.
template <typename AccT>
__device__ __forceinline__ bool acc_add_first(AccT* acc, int slot, int add, bool& ovf);
template <>
__device__ __forceinline__ bool acc_add_first<int32_t>(int32_t* acc, int slot, int add, bool&) {
  return atomicAdd(&acc[slot], add) == 0;
}
template <>
__device__ __forceinline__ bool acc_add_first<uint16_t>(uint16_t* acc, int slot, int add, bool& ovf) {
  const int sh = (slot & 1) * 16;
  const uint32_t old = atomicAdd(reinterpret_cast<uint32_t*>(acc) + (slot >> 1), uint32_t(add) << sh);
  const uint32_t old16 = (old >> sh) & 0xFFFFu;
  ovf |= old16 + uint32_t(add) > 0xFFFFu;
  return old16 == 0;
}

}  // namespace lr

#include "sparse_rows.cuh"  // the row kernel (dense batches)

namespace lr {

// Flat kernel: flattened posting slots + shared-memory atomics (the round-1 design).  It serves SPARSE batches — short
// posting runs, where a row of the row kernel would be mostly empty lanes — and stays selectable for same-box A/B runs.
template <int BD, int NB, typename AccT>
__global__ void __launch_bounds__(SS_MAX_WARPS * 32, 1)
sparse_score_kernel(const SSParams p) {
  if (sizeof(AccT) == 4 && p.overflow && ld_relaxed_u32(p.overflow) == 0) return;  // the 16-bit pass was exact
  if (ss_regime_skip(p)) return;
  extern __shared__ __align__(16) uint8_t ss_smem[];
  const uint32_t full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t lt = lanemask_lt();
  uint8_t* wbase = ss_smem + size_t(warp) * p.warp_bytes;
  AccT* acc = reinterpret_cast<AccT*>(wbase);
  uint64_t* list = reinterpret_cast<uint64_t*>(wbase + size_t(BD) * sizeof(AccT));
  uint32_t* hist = reinterpret_cast<uint32_t*>(list + p.cap);
  uint16_t* touched = reinterpret_cast<uint16_t*>(hist + 256);

  for (int i = lane; i < BD; i += 32) acc[i] = 0;
  __syncwarp();

  const uint32_t n_units = uint32_t(p.Q * p.S);
  for (;;) {
    uint32_t u = 0;
    if (lane == 0) u = atomicAdd(p.next_unit, 1u);
    u = __shfl_sync(full, u, 0);
    if (u >= n_units) break;
    const int64_t q = u / uint32_t(p.S);
    const int s = int(u % uint32_t(p.S));
    const int b0 = int((int64_t(s) * p.nblk) / p.S);
    const int b1 = int((int64_t(s + 1) * p.nblk) / p.S);
    const int qt0 = p.q_indptr[q];
    const int nterms = p.q_indptr[q + 1] - qt0;
    const int f_row = p.filter.on ? filter_row(p.filter, q) : FILTER_ALL;  // a unit is one query: warp-uniform
    // a step = (document block, chunk of 32 query terms); lane t owns term t of the chunk.  Queries of <= 32 terms (the
    // normal case) walk their blockptr rows with a two-block-ahead prefetch; longer ones fetch the pointers per step.
    const int nchunks = nterms > 32 ? (nterms + 31) >> 5 : 1;
    const bool one_chunk = nchunks == 1;
    const int nsteps = (b1 - b0) * nchunks;
    uint32_t n = 0;                // entries in `list` (warp-uniform)
    uint64_t thr = 0xFFFFFFFFull;  // candidates need key > thr; every score-0 key is <= this
    uint32_t ntouch = 0;           // accumulators touched in the current block (warp-uniform)
    bool ovf = false;

    const uint32_t* bp_row = nullptr;
    int64_t post_base = 0;
    uint32_t lo = 0, hi = 0, nxt = 0;
    int w_cur = 0;  // this lane's term weight for the batch waiting in registers
    if (one_chunk && lane < nterms) {
      const int t = p.q_tok[qt0 + lane];
      const int w = p.q_cnt[qt0 + lane];
      if (t >= 0 && t < p.V && w > 0) {  // terms with a count <= 0 contribute nothing
        bp_row = p.blockptr + int64_t(t) * (p.nblk + 1);
        post_base = p.post_indptr[t];
        w_cur = w;
        lo = bp_row[b0];
        hi = bp_row[b0 + 1];
        nxt = (b0 + 2 <= p.nblk) ? bp_row[b0 + 2] : hi;
      }
    }
    // flatten state of the batch waiting in registers, and the batch itself (NB postings per lane)
    int total = 0, pre = 0;
    int64_t rel = 0;  // posting index of flattened position j inside this lane's term = rel + j
    int doc[NB], imp[NB], tl[NB];
    int pb = b0, pc = 0;  // step the next load phase fetches
    int ab = b0, ac = 0;  // step of the waiting batch
    uint32_t floor_s = 0;

    // largest l in [0, 32) with pre[l] <= j (lanes past the last term hold pre == total > j)
    auto find_term = [&](int j) {
      int l = 0;
#pragma unroll
      for (int step = 16; step >= 1; step >>= 1) {
        const int pv = __shfl_sync(full, pre, l + step);
        if (pv <= j) l += step;
      }
      return l;
    };
    // the first add that finds 0 records the slot
    auto note_first = [&](bool first, int slot) {
      const uint32_t fm = __ballot_sync(full, first);
      const uint32_t tpos = ntouch + __popc(fm & lt);
      if (first && tpos < SS_TOUCH_CAP) touched[tpos] = uint16_t(slot);
      ntouch += __popc(fm);
    };

    for (int e = -1; e < nsteps; ++e) {
      if (e >= 0) {
        // ---- accumulate the waiting batch: all atomics first, then the first-touch bookkeeping
        const int d0 = ab * BD;
        if (ac == 0 && p.S > 1) floor_s = ld_relaxed_u32(p.floor_q + q);  // consumed by the visit
        bool fst[NB];
        int slot[NB];
#pragma unroll
        for (int i = 0; i < NB; ++i) {
          fst[i] = false;
          slot[i] = doc[i] - d0;
          if (i * 32 < total) {  // warp-uniform
            const int add = __shfl_sync(full, w_cur, tl[i]) * imp[i];
            if (add != 0) fst[i] = acc_add_first<AccT>(acc, slot[i], add, ovf);
          }
        }
#pragma unroll
        for (int i = 0; i < NB; ++i)
          if (i * 32 < total) note_first(fst[i], slot[i]);
        // postings beyond the register batch (long posting runs): direct
        for (int j0 = 32 * NB; j0 < total; j0 += 32) {
          const int j = min(j0 + lane, total - 1);
          const int l = find_term(j);
          const int64_t idx = __shfl_sync(full, rel, l) + j;
          const int wl = __shfl_sync(full, w_cur, l);
          const int sl = __ldg(p.post_doc + idx) - d0;
          const int add = j0 + lane < total ? wl * int(__ldg(p.post_imp + idx)) : 0;
          bool first = false;
          if (add != 0) first = acc_add_first<AccT>(acc, sl, add, ovf);
          note_first(first, sl);
        }
      }
      if (e + 1 < nsteps) {
        // ---- load phase of the next step: its postings are in flight while the current block is visited
        int cnt = 0;
        int64_t start = 0;
        if (one_chunk) {
          if (bp_row) {
            start = post_base + lo;
            cnt = int(hi - lo);
            lo = hi;
            hi = nxt;
            if (pb + 3 <= p.nblk && pb + 2 < b1) nxt = bp_row[pb + 3];  // consumed two blocks from now
          }
        } else {
          const int i = pc * 32 + lane;
          w_cur = 0;
          if (i < nterms) {
            const int t = p.q_tok[qt0 + i];
            const int wi = p.q_cnt[qt0 + i];
            if (t >= 0 && t < p.V && wi > 0) {
              const uint32_t* bp = p.blockptr + int64_t(t) * (p.nblk + 1) + pb;
              const uint32_t l2 = bp[0], h2 = bp[1];
              start = p.post_indptr[t] + l2;
              cnt = int(h2 - l2);
              w_cur = wi;
            }
          }
        }
        int incl = cnt;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const int t = __shfl_up_sync(full, incl, off);
          if (lane >= off) incl += t;
        }
        total = __shfl_sync(full, incl, 31);
        pre = incl - cnt;
        rel = start - pre;
#pragma unroll
        for (int i = 0; i < NB; ++i) {
          if (i * 32 < total) {  // warp-uniform
            const int j = min(i * 32 + lane, total - 1);  // lanes past the end repeat the last posting's address
            const int l = find_term(j);
            const int64_t idx = __shfl_sync(full, rel, l) + j;
            tl[i] = l;
            doc[i] = __ldg(p.post_doc + idx);
            imp[i] = i * 32 + lane < total ? int(__ldg(p.post_imp + idx)) : 0;
          }
        }
        if (++pc == nchunks) {
          pc = 0;
          ++pb;
        }
      }
      if (e >= 0) {
        if (ac == nchunks - 1) {
          // ---- visit the touched accumulators of block ab (or all of them when the touched list overflowed)
          __syncwarp();
          const int d0 = ab * BD;
          const bool dense = ntouch > SS_TOUCH_CAP;
          const uint32_t n_visit = dense ? uint32_t(BD) : ntouch;
          for (uint32_t i0 = 0; i0 < n_visit; i0 += 32) {
            const uint32_t i = min(i0 + lane, n_visit - 1);
            const int sl = dense ? int(i) : int(touched[i]);
            const int sc = i0 + lane < n_visit ? int(acc[sl]) : 0;
            if (sc != 0) acc[sl] = 0;
            const uint64_t key = make_key(uint32_t(sc), uint32_t(d0 + sl));
            bool pass = uint32_t(sc) >= floor_s && key > thr;  // key > thr implies sc > 0
            if (pass && p.filter.on) pass = filter_allows(p.filter, f_row, d0 + sl);  // (d0 + sl: shard-local id)
            uint32_t pm = __ballot_sync(full, pass);
            while (pm) {
              const uint32_t room = uint32_t(p.cap) - n;
              const uint32_t rank = __popc(pm & lt);
              if (pass && rank < room) {
                list[n + rank] = key;
                pass = false;
              }
              n += min(uint32_t(__popc(pm)), room);
              __syncwarp();
              if (n == uint32_t(p.cap)) {
                thr = warp_cut_topk(list, &n, p.k, hist);
                if (p.S > 1 && lane == 0) atomicMax(p.floor_q + q, key_hi(thr));
                pass = pass && key > thr;
              }
              pm = __ballot_sync(full, pass);
            }
          }
          ntouch = 0;
          __syncwarp();
          ac = 0;
          ++ab;
        } else {
          ++ac;
        }
      }
    }
    if (sizeof(AccT) == 2 && __any_sync(full, ovf) && lane == 0) atomicOr(p.overflow, 1u);
    // ---- unit result
    uint64_t* dst = p.cand + (int64_t(s) * p.Q + q) * p.cap;
    for (uint32_t i = lane; i < n; i += 32) dst[i] = list[i];
    if (lane == 0) p.counts[int64_t(s) * p.Q + q] = int32_t(n);
    __syncwarp();
  }
}

// Postings and terms of the whole query batch -> regime words (see SSParams::regime).  One thread per query.
__global__ void sparse_density_kernel(const int32_t* __restrict__ q_indptr, const int32_t* __restrict__ q_tok,
                                      const int32_t* __restrict__ q_cnt, int64_t Q, const int64_t* __restrict__ post_indptr,
                                      int64_t V, uint32_t* regime) {
  const int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  unsigned long long postings = 0;
  uint32_t terms = 0;
  if (q < Q) {
    for (int i = q_indptr[q]; i < q_indptr[q + 1]; ++i) {
      const int t = q_tok[i];
      if (t >= 0 && t < V && q_cnt[i] > 0) {
        postings += static_cast<unsigned long long>(post_indptr[t + 1] - post_indptr[t]);
        ++terms;
      }
    }
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    postings += __shfl_xor_sync(0xFFFFFFFFu, postings, off);
    terms += __shfl_xor_sync(0xFFFFFFFFu, terms, off);
  }
  if ((threadIdx.x & 31) == 0 && terms) {
    atomicAdd(reinterpret_cast<unsigned long long*>(regime), postings);
    atomicAdd(regime + 2, terms);
  }
}

__global__ void build_blockptr_kernel(const int64_t* __restrict__ post_indptr, const int32_t* __restrict__ post_doc,
                                      int64_t V, int nblk, int block_docs, uint32_t* __restrict__ blockptr) {
  const int64_t total = V * int64_t(nblk + 1);
  for (int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += int64_t(gridDim.x) * blockDim.x) {
    const int64_t t = e / (nblk + 1);
    const int b = int(e % (nblk + 1));
    const int64_t lo0 = post_indptr[t], hi0 = post_indptr[t + 1];
    const int64_t bound = int64_t(b) * block_docs;
    int64_t lo = lo0, hi = hi0;  // first index with doc >= bound
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (int64_t(post_doc[mid]) < bound) lo = mid + 1; else hi = mid;
    }
    blockptr[e] = uint32_t(lo - lo0);
  }
}

static_assert(SR_ACC_BYTES / 4 >= SS_BLOCK_DOCS, "the row kernel steps over whole index blocks (its 32-bit pass too)");

struct SSPlan {
  int nblk, cap;
  bool rows, flat;  // which kernels a call launches
  // [0] / [1] = flat kernel with 16-bit / int32 accumulators, [2] / [3] = row kernel with 16-bit / 32-bit accumulators
  int warps[4], warp_bytes[4], grid[4];
  size_t smem[4];
  int S_flat, S_rows, S;  // splits per query of each kernel; S = the larger one = candidate lists per query
  size_t off_counts, off_floor, off_thr, off_cand, off_merge, merge_bytes, total_bytes;
};

static SSPlan ss_plan(int64_t Q, int64_t N, int k, const Knobs& kn) {
  SSPlan pl{};
  pl.nblk = int((N + SS_BLOCK_DOCS - 1) / SS_BLOCK_DOCS);
  int cap = k + (k / 2 > 156 ? k / 2 : 156);  // k = 100 -> 256
  pl.cap = (cap + 31) / 32 * 32;
  const int G = sm_count();
  // by regime (dense batches: row kernel, sparse batches: flat kernel; decided on the device from the batch's mean
  // posting run, both kernels are launched and the other one returns at once), or the one kernel the knob forces
  pl.rows = kn.sparse_kernel != 1;
  pl.flat = kn.sparse_kernel != 3;
  for (int m = 0; m < 4; ++m) {
    const bool row = m >= 2;
    pl.warp_bytes[m] = row ? SR_ACC_BYTES + 32 * 16 + pl.cap * 8 + 256 * 4 + 16
                           : SS_BLOCK_DOCS * ((m & 1) ? 4 : 2) + pl.cap * 8 + 256 * 4 + SS_TOUCH_CAP * 2;
    const int max_warps = row ? SR_MAX_WARPS : SS_MAX_WARPS;
    const int warps = int((size_t(227) * 1024 - 1024) / size_t(pl.warp_bytes[m]));
    pl.warps[m] = warps > max_warps ? max_warps : warps;
    pl.smem[m] = size_t(pl.warps[m]) * pl.warp_bytes[m];
  }
  // enough units to balance the dynamic hand-out (8 per warp), at most one unit per document block and at most 64
  // lists per query for the merge
  auto clampS = [&](int64_t S) {
    if (S > 64) S = 64;
    if (S > pl.nblk) S = pl.nblk;
    return int(S < 1 ? 1 : S);
  };
  pl.S_flat = clampS((8 * int64_t(G) * pl.warps[kn.sparse_acc32 ? 1 : 0] + Q - 1) / Q);
  {
    // The row kernel hands units out split-major, so the workers running together read the same slice of the index;
    // more splits = a smaller slice (the posting runs of frequent terms stay in L2), as long as a unit keeps >= 4 steps.
    int64_t S = (8 * int64_t(G) * pl.warps[2] + Q - 1) / Q;
    const int64_t steps = (N + SR_ACC_BYTES / 2 - 1) / (SR_ACC_BYTES / 2);
    if (S < steps / 4) S = steps / 4;
    pl.S_rows = clampS(S);
  }
  pl.S = !pl.rows ? pl.S_flat : (!pl.flat ? pl.S_rows : (pl.S_flat > pl.S_rows ? pl.S_flat : pl.S_rows));
  for (int m = 0; m < 4; ++m) {
    const int64_t units = Q * (m >= 2 ? pl.S_rows : pl.S_flat);
    const int64_t ctas = (units + pl.warps[m] - 1) / (pl.warps[m] > 0 ? pl.warps[m] : 1);
    pl.grid[m] = int(ctas < G ? ctas : G);
  }
  auto align = [](size_t x) { return (x + 255) / 256 * 256; };
  pl.off_counts = 0;
  // control block, zeroed per call together with the counts: floor_q [4][Q] (one per kernel pass), 4 unit counters,
  // overflow flag, regime words; then (row kernel) the finished-unit thresholds of its two passes
  pl.off_floor = align(size_t(pl.S) * Q * 4);
  pl.off_thr = align(pl.off_floor + 4 * size_t(Q) * 4 + 256);
  pl.off_cand = align(pl.off_thr + (pl.rows && pl.S_rows > 1 ? 2 * size_t(Q) * pl.S_rows * 8 : 0));
  pl.off_merge = align(pl.off_cand + size_t(pl.S) * Q * pl.cap * 8);
  pl.merge_bytes = topk_merge_scratch_bytes(pl.S, Q, pl.cap, k);
  pl.total_bytes = align(pl.off_merge + pl.merge_bytes);
  return pl;
}

template <typename AccT>
static int ss_launch(const SSParams& p, const SSPlan& pl, cudaStream_t st) {
  const int m = sizeof(AccT) == 4 ? 1 : 0;
  auto kern = sparse_score_kernel<SS_BLOCK_DOCS, SS_NB, AccT>;
  int rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), 227 * 1024);
  if (rc) return rc;
  kern<<<pl.grid[m], pl.warps[m] * 32, pl.smem[m], st>>>(p);
  LR_LAUNCH_CHECK();
  return LR_OK;
}

template <typename AccT>
static int sr_launch(const SSParams& p, const SSPlan& pl, cudaStream_t st) {
  const int m = sizeof(AccT) == 4 ? 3 : 2;
  auto kern = p.filter.on ? sparse_score_rows_kernel<SR_ACC_BYTES, AccT, true> : sparse_score_rows_kernel<SR_ACC_BYTES, AccT, false>;
  int rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), 227 * 1024);
  if (rc) return rc;
  kern<<<pl.grid[m], pl.warps[m] * 32, pl.smem[m], st>>>(p);
  LR_LAUNCH_CHECK();
  return LR_OK;
}

}  // namespace lr

using namespace lr;

extern "C" int lr_sparse_block_docs(void) { return SS_BLOCK_DOCS; }

extern "C" int lr_sparse_build_blockptr(const int64_t* post_indptr, const int32_t* post_doc, int64_t V, int64_t N,
                                        uint32_t* blockptr, void* stream) {
  LR_CHECK_ARG(post_indptr && blockptr && V >= 1 && N >= 1, "build_blockptr: bad arguments");
  const int bd = SS_BLOCK_DOCS;
  const int nblk = int((N + bd - 1) / bd);
  const int64_t total = V * int64_t(nblk + 1);
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  build_blockptr_kernel<<<unsigned(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(post_indptr, post_doc, V, nblk,
                                                                                        bd, blockptr);
  LR_LAUNCH_CHECK();
  return LR_OK;
}

// Planner introspection (host only; CPU tests): out[16] = block_docs, index blocks, list capacity, flat kernel launched,
// row kernel launched, splits of the flat kernel, splits of the row kernel, lists per query, workers per CTA and dynamic
// shared memory of the flat 16-bit / flat int32 / row 16-bit / row 32-bit launches (4 x 2), workspace bytes, step docs
extern "C" int lr_sparse_score_plan(int64_t Q, int64_t N, int k, int64_t* out) {
  LR_CHECK_ARG(out && Q >= 1 && N >= 1 && k >= 1, "sparse_score_plan: bad arguments");
  const SSPlan pl = ss_plan(Q, N, k, knobs());
  int i = 0;
  out[i++] = SS_BLOCK_DOCS; out[i++] = pl.nblk; out[i++] = pl.cap; out[i++] = pl.flat; out[i++] = pl.rows;
  out[i++] = pl.S_flat; out[i++] = pl.S_rows; out[i++] = pl.S;
  for (int m = 0; m < 4; ++m) {
    out[i++] = pl.warps[m];
  }
  for (int m = 0; m < 2; ++m) out[i++] = int64_t(pl.smem[m * 2]);  // flat 16-bit, row 16-bit
  out[i++] = int64_t(pl.total_bytes);
  out[i++] = SR_ACC_BYTES / 2;
  return LR_OK;
}

extern "C" size_t lr_sparse_score_workspace_bytes(int64_t Q, int64_t N, int k) {
  if (Q < 1 || N < 1 || k < 1) return 0;
  return ss_plan(Q, N, k, knobs()).total_bytes;
}

// The unfiltered and filtered entry points share this path (null bitmaps = no filter).
static int sparse_score_run(const int32_t* q_indptr, const int32_t* q_tok, const int32_t* q_cnt, int64_t Q,
                            const int64_t* post_indptr, const int32_t* post_doc, const uint16_t* post_imp,
                            const uint32_t* blockptr, int64_t V, int64_t N, int64_t id_offset, int k,
                            float* out_scores, int64_t* out_ids, uint64_t* out_keys, const uint32_t* live,
                            const uint32_t* allow, int64_t ld_words, int n_filters, const int32_t* q_filter,
                            void* workspace, size_t ws_bytes, void* stream) {
  LR_CHECK_ARG(q_indptr && post_indptr && blockptr, "sparse_score: null pointer");
  LR_CHECK_ARG(Q >= 1 && N >= 1 && V >= 1, "sparse_score: Q, N, V must be >= 1");
  LR_CHECK_ARG(N < (int64_t(1) << 31), "sparse_score: N must be < 2^31 per shard");
  LR_CHECK_ARG(k >= 1 && k <= 1024, "sparse_score: k (%d) must be in [1, 1024]", k);
  LR_CHECK_ARG(id_offset >= 0 && id_offset + N <= (int64_t(1) << 32) - 2, "sparse_score: id_offset + N must stay below 2^32");
  LR_CHECK_ARG(out_scores || out_ids || out_keys, "sparse_score: no output requested");
  DocFilter flt;
  if (int frc = make_doc_filter(live, allow, ld_words, n_filters, q_filter, id_offset, N, flt)) return frc;
  const Knobs& kn = knobs();
  SSPlan pl = ss_plan(Q, N, k, kn);
  LR_CHECK_ARG(Q * int64_t(pl.S) < (int64_t(1) << 31), "sparse_score: too many (query, block range) units");
  for (int m = 0; m < 4; ++m)
    LR_CHECK_ARG(pl.warps[m] >= 1, "sparse_score: k (%d) leaves no shared memory for a worker", k);
  if (!workspace || ws_bytes < pl.total_bytes || (uintptr_t(workspace) & 255)) {
    set_error("sparse_score: workspace too small or misaligned (%zu given, %zu needed)", ws_bytes, pl.total_bytes);
    return LR_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  SSParams p{};
  p.q_indptr = q_indptr; p.q_tok = q_tok; p.q_cnt = q_cnt; p.Q = Q;
  p.post_indptr = post_indptr; p.post_doc = post_doc; p.post_imp = post_imp; p.blockptr = blockptr;
  p.V = V; p.N = N; p.nblk = pl.nblk; p.k = k; p.cap = pl.cap; p.bd = SS_BLOCK_DOCS;
  p.filter = flt;
  p.counts = reinterpret_cast<int32_t*>(ws + pl.off_counts);
  p.cand = reinterpret_cast<uint64_t*>(ws + pl.off_cand);
  // counts (a kernel that sits the call out, or runs fewer splits, leaves empty lists) + control block + unit thresholds
  LR_CUDA(cudaMemsetAsync(ws, 0, pl.off_cand, st));
  uint32_t* ctl = reinterpret_cast<uint32_t*>(ws + pl.off_floor);
  uint32_t* next4 = ctl + 4 * Q;
  uint32_t* regime = next4 + 8;  // 8-byte aligned (off_floor is 256-aligned, 16 * Q + 32 bytes further)
  p.overflow = next4 + 4;
  int rc = LR_OK;
  const ProfileEvents pe = profile_events();  // lr_set_profile_events: bracket the scoring kernels (not the merge)
  if (pe.begin && pe.end) LR_CUDA(cudaEventRecord(pe.begin, st));
  if (pl.rows && pl.flat) {
    sparse_density_kernel<<<unsigned((Q + 255) / 256), 256, 0, st>>>(q_indptr, q_tok, q_cnt, Q, post_indptr, V, regime);
    LR_LAUNCH_CHECK();
    p.regime = regime;
    const int64_t steps = (N + SR_ACC_BYTES / 2 - 1) / (SR_ACC_BYTES / 2);
    p.dense_thresh = uint32_t(SS_DENSE_RUN * steps);
  }
  uint64_t* unit_thr = (pl.rows && pl.S_rows > 1) ? reinterpret_cast<uint64_t*>(ws + pl.off_thr) : nullptr;
  // Per kernel: an optimistic pass with 16-bit accumulators (exact unless a document's score would exceed 65535: flag),
  // then a pass with 32-bit accumulators that returns at once unless the flag is set (kn.sparse_acc32: that pass alone).
  if (pl.flat) {
    p.S = pl.S_flat;
    p.want_dense = 0;
    p.unit_thr = nullptr;
    if (!kn.sparse_acc32) {
      p.floor_q = ctl;
      p.next_unit = next4;
      p.warp_bytes = pl.warp_bytes[0];
      if ((rc = ss_launch<uint16_t>(p, pl, st)) != LR_OK) return rc;
    }
    SSParams p2 = p;
    if (kn.sparse_acc32) p2.overflow = nullptr;
    p2.floor_q = ctl + Q;
    p2.next_unit = next4 + 1;
    p2.warp_bytes = pl.warp_bytes[1];
    if ((rc = ss_launch<int32_t>(p2, pl, st)) != LR_OK) return rc;
  }
  if (pl.rows) {
    p.S = pl.S_rows;
    p.want_dense = 1;
    if (!kn.sparse_acc32) {
      p.floor_q = ctl + 2 * Q;
      p.next_unit = next4 + 2;
      p.warp_bytes = pl.warp_bytes[2];
      p.unit_thr = unit_thr;
      if ((rc = sr_launch<uint16_t>(p, pl, st)) != LR_OK) return rc;
    }
    SSParams p2 = p;
    if (kn.sparse_acc32) p2.overflow = nullptr;
    p2.floor_q = ctl + 3 * Q;
    p2.next_unit = next4 + 3;
    p2.warp_bytes = pl.warp_bytes[3];
    p2.unit_thr = unit_thr ? unit_thr + size_t(Q) * pl.S_rows : nullptr;
    if ((rc = sr_launch<uint32_t>(p2, pl, st)) != LR_OK) return rc;
  }
  if (pe.begin && pe.end) LR_CUDA(cudaEventRecord(pe.end, st));
  if (kn.sparse_debug) {  // diagnostics: regime words and the overflow flag
    uint32_t host[12] = {0};
    LR_CUDA(cudaStreamSynchronize(st));
    LR_CUDA(cudaMemcpy(host, next4, sizeof(host), cudaMemcpyDeviceToHost));
    const uint32_t* rg = host + (regime - next4);
    fprintf(stderr, "lr_b200 sparse_score: S flat %d rows %d, 16-bit overflow %u, batch postings %llu over %u terms, dense from %u\n",
            pl.S_flat, pl.S_rows, host[4], (unsigned long long)((uint64_t(rg[1]) << 32) | rg[0]), rg[2], p.dense_thresh);
  }
  return topk_merge_two_level(p.cand, p.counts, pl.S, Q, Q, pl.cap, k, LR_SCORE_U32, id_offset, out_scores, out_ids,
                              out_keys, k, ws + pl.off_merge, pl.merge_bytes, st);
}

extern "C" int lr_sparse_score_topk(const int32_t* q_indptr, const int32_t* q_tok, const int32_t* q_cnt, int64_t Q,
                                    const int64_t* post_indptr, const int32_t* post_doc, const uint16_t* post_imp,
                                    const uint32_t* blockptr, int64_t V, int64_t N, int64_t id_offset, int k,
                                    float* out_scores, int64_t* out_ids, uint64_t* out_keys, void* workspace,
                                    size_t ws_bytes, void* stream) {
  return sparse_score_run(q_indptr, q_tok, q_cnt, Q, post_indptr, post_doc, post_imp, blockptr, V, N, id_offset, k,
                          out_scores, out_ids, out_keys, nullptr, nullptr, 0, 0, nullptr, workspace, ws_bytes, stream);
}

extern "C" int lr_sparse_score_topk_filtered(const int32_t* q_indptr, const int32_t* q_tok, const int32_t* q_cnt,
                                             int64_t Q, const int64_t* post_indptr, const int32_t* post_doc,
                                             const uint16_t* post_imp, const uint32_t* blockptr, int64_t V, int64_t N,
                                             int64_t id_offset, int k, float* out_scores, int64_t* out_ids,
                                             uint64_t* out_keys, const uint32_t* live, const uint32_t* allow,
                                             int64_t ld_words, int n_filters, const int32_t* q_filter, void* workspace,
                                             size_t ws_bytes, void* stream) {
  return sparse_score_run(q_indptr, q_tok, q_cnt, Q, post_indptr, post_doc, post_imp, blockptr, V, N, id_offset, k,
                          out_scores, out_ids, out_keys, live, allow, ld_words, n_filters, q_filter, workspace,
                          ws_bytes, stream);
}
