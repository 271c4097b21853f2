// sparse_rows.cuh — K4, row kernel (round 2; dense batches): the same gather-accumulate as sparse_score_kernel without a
// single shared-memory atomic.
//
// Why: the accumulator kernel of round 1 issues one shared-memory atomicAdd per posting.  Scattered ATOMS retire at
// about one lane every two cycles per SM, so 3.6e8 postings (10k uniform queries over a 1.1M-document shard) cost
// >= 2.5 ms and 4.8e10 postings (the Zipf workload) >= 340 ms in atomics alone — 60-70 % of what was measured.
//
// How: a ROW is 32 consecutive postings of ONE term.  The postings of a term carry strictly ascending document ids, so
// the 32 lanes of a row hit 32 different accumulators and a plain LDS / IADD / STS read-modify-write is exact; rows are
// retired one after the other by the same warp (shared memory is processed in order, __syncwarp between rows), and the
// accumulators are private to the warp, so no other writer exists.  Everything else keeps the round-1 structure:
// warp-granular workers without block barriers, units = (query, range of document blocks) handed out dynamically,
// lane t owns query term t and walks its blockptr row two steps ahead, the loads of the next batch of rows are issued
// before the current batch is accumulated, 16-bit accumulators with an int32 fallback launch.
//
// Candidates are taken on the RUNNING sum: right after the read-modify-write a lane compares the new sum with the
// unit's score threshold; a sum only grows, so a document whose final score reaches the threshold is seen with exactly
// that score at its last posting.  A document that passes more than once is replaced in the list in place (it can only
// be listed when its previous sum already met the threshold, which is rare enough for a warp-wide search).  No touched
// list, no second walk: at the end of a step the accumulator block is cleared with 16-byte stores.
//
// Long posting runs (frequent terms: the Zipf head) take a second path: a batch of NB full rows of ONE term has no two
// postings of the same document, so its read-modify-writes are issued as loads, then adds, then stores (no chain
// from row to row), the addresses come from one base pointer with immediate offsets, and one vote covers the batch.
//
// Units of one query are chained: unit (split s, query q) starts from the candidate list and threshold that unit
// (s - 1, q) left behind when that unit has already finished (always, once there are more queries than workers), so the
// threshold a posting is compared with is the running k-th best of everything scored so far for that query instead of
// the k-th best of one slice.  An inherited list is struck from the merge (its count is zeroed).
//
// Units are ordered split-major (all queries for one range of document blocks, then the next range), so the workers
// running at any moment read the same slice of the index and the posting runs of frequent terms are served from L2.
#pragma once

namespace lr {

constexpr int SR_NB = 8;          // rows whose loads are in flight together, per warp (x2: the next batch is issued first)
constexpr int SR_MAX_WARPS = 11;  // workers per CTA (shared memory: acc + list + hist + table per warp)
// accumulator bytes per worker: 8192 documents per step with 16-bit accumulators (32 / 64 KB steps were slower in both
// regimes: fewer resident warps, DESIGN.md K4)
constexpr int SR_ACC_BYTES = 16 * 1024;

// A batch of rows in flight.  General rows: doc = x[i], impact = x[NB + i], weight = x[2 NB + i] (0 for lanes past the
// end of the run).  Long run (w != 0): NBF = 3 NB / 2 full rows of one term, doc = x[i], impact = x[NBF + i].
template <int NB> struct RowBatch {
  uint32_t x[3 * NB];
  int nb;      // rows in the batch (warp-uniform); 0 = no more work in this unit
  int d0;      // first document of the step the batch belongs to
  uint32_t w;  // != 0: long-run batch of this weight
};

// Candidate list state of a worker (warp-uniform; shared memory, so that the candidate path can be an out-of-line call
// instead of sixteen inlined copies in the row loops).
struct SRList {
  uint64_t thr;     // candidates need key > thr
  uint32_t n;       // entries in the list
  uint32_t min_sc;  // max(global floor of the step, score part of thr, 1): the one compare every posting pays
};

__device__ __forceinline__ uint64_t ld_acquire_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Slow part of the candidate path: replacement of listed documents, appends that fill the list, cuts.
static __device__ __noinline__ void sr_candidate_slow(uint64_t* list, uint32_t* hist, SRList* st, uint32_t* floor_q, int cap,
                                                     int k, bool pass, uint64_t key, uint32_t old) {
  const uint32_t full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const uint32_t lt = lanemask_lt();
  uint32_t n = st->n, min_sc = st->min_sc;
  uint64_t thr = st->thr;
  // a document whose previous sum met the threshold may be listed: replace its entry in place
  uint32_t dm = __ballot_sync(full, pass && old >= min_sc);
  while (dm) {
    const int r = __ffs(dm) - 1;
    dm &= dm - 1;
    const uint64_t kr = __shfl_sync(full, key, r);
    bool found = false;
    for (uint32_t i0 = 0; i0 < n && !found; i0 += 32) {
      const uint32_t i = i0 + lane;
      const bool hit = i < n && uint32_t(list[i]) == uint32_t(kr);
      if (hit) list[i] = kr;
      found = __any_sync(full, hit);
    }
    if (found && lane == r) pass = false;
  }
  __syncwarp();
  uint32_t pm = __ballot_sync(full, pass);
  while (pm) {
    const uint32_t room = uint32_t(cap) - n;
    const uint32_t rank = __popc(pm & lt);
    if (pass && rank < room) {
      list[n + rank] = key;
      pass = false;
    }
    n += min(uint32_t(__popc(pm)), room);
    __syncwarp();
    if (n == uint32_t(cap)) {
      thr = warp_cut_topk(list, &n, k, hist);
      if (floor_q && lane == 0) atomicMax(floor_q, key_hi(thr));
      min_sc = max(min_sc, key_hi(thr));
      pass = pass && key > thr;
    }
    pm = __ballot_sync(full, pass);
  }
  __syncwarp();
  if (lane == 0) {
    st->n = n;
    st->thr = thr;
    st->min_sc = min_sc;
  }
  __syncwarp();
}

// The unit's document filter in the row kernel's filtered instantiation: global id of local document 0, the `live`
// bitmap and the query's `allow` row (null = none), or deny = 1 for a query whose filter row is out of range.
struct SRFilter {
  const uint32_t* live;
  const uint32_t* arow;
  int64_t base;
  int deny;
};
__device__ __forceinline__ bool sr_allowed(const SRFilter& f, uint32_t docid) {
  if (f.deny) return false;
  const int64_t id = f.base + docid;
  const uint32_t bit = 1u << (id & 31);
  return (!f.live || (f.live[id >> 5] & bit)) && (!f.arow || (f.arow[id >> 5] & bit));
}

// Lanes whose new running sum `sc` met the score threshold (the caller's vote said at least one did).  Returns the
// (possibly raised) score threshold.  All 32 lanes call.  Fast path: nobody survives the exact test, or the survivors
// are new to the list and fit.  The filtered instantiation passes the unit's SRFilter (the unfiltered one keeps its
// argument list): a document the query may not return never passes, so it is never listed — the in-place replacement of
// sr_candidate_slow only ever meets allowed documents, and every cut, floor and inherited threshold is taken over
// allowed documents.  docid is the shard-local id.
template <typename... Flt>
static __device__ __noinline__ uint32_t sr_candidate(uint64_t* list, uint32_t* hist, SRList* st, uint32_t* floor_q, int cap,
                                                    int k, uint32_t sc, uint32_t old, uint32_t docid, Flt... flt) {
  const uint32_t full = 0xFFFFFFFFu;
  const uint32_t n = st->n, min_sc = st->min_sc;
  const uint64_t key = make_key(sc, docid);
  bool pass = sc >= min_sc && key > st->thr;
  if constexpr (sizeof...(Flt) > 0) {
    if (pass) pass = sr_allowed(flt..., docid);
  }
  const uint32_t pm = __ballot_sync(full, pass);
  if (pm == 0) return min_sc;
  const uint32_t c = __popc(pm);
  if (n + c < uint32_t(cap) && !__any_sync(full, pass && old >= min_sc)) {
    if (pass) list[n + __popc(pm & lanemask_lt())] = key;
    __syncwarp();
    if ((threadIdx.x & 31) == 0) st->n = n + c;
    __syncwarp();
    return min_sc;
  }
  sr_candidate_slow(list, hist, st, floor_q, cap, k, pass, key, old);
  return st->min_sc;
}

// ACC_BYTES of accumulators per warp: STEP_DOCS = ACC_BYTES / sizeof(AccT) documents per step.
// FILTERED: the instantiation launched when p.filter.on (the unfiltered one is the kernel without any filter code).
template <int ACC_BYTES, typename AccT, bool FILTERED>
__global__ void __launch_bounds__(SR_MAX_WARPS * 32, 1)
sparse_score_rows_kernel(const SSParams p) {
  if (sizeof(AccT) == 4 && p.overflow && ld_relaxed_u32(p.overflow) == 0) return;  // the 16-bit pass was exact
  if (ss_regime_skip(p)) return;  // a sparse batch (short posting runs) is the flat kernel's
  constexpr int NB = SR_NB;
  constexpr int NBF = 3 * NB / 2;  // rows of a long-run batch (same registers: no per-lane weights)
  constexpr int STEP_DOCS = ACC_BYTES / int(sizeof(AccT));
  extern __shared__ __align__(16) uint8_t ss_smem[];
  const uint32_t full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* wbase = ss_smem + size_t(warp) * p.warp_bytes;
  AccT* acc = reinterpret_cast<AccT*>(wbase);
  uint4* tab = reinterpret_cast<uint4*>(wbase + ACC_BYTES);  // per term of the step being loaded: run base, end, weight
  uint64_t* list = reinterpret_cast<uint64_t*>(wbase + ACC_BYTES + 32 * 16);
  uint32_t* hist = reinterpret_cast<uint32_t*>(list + p.cap);
  SRList* st = reinterpret_cast<SRList*>(hist + 256);
  const int G = STEP_DOCS / p.bd;  // index blocks per step (host guarantees >= 1)

  auto clear_acc = [&]() {
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    uint4* a4 = reinterpret_cast<uint4*>(acc);
#pragma unroll 8
    for (int i = lane; i < ACC_BYTES / 16; i += 32) a4[i] = z;
    __syncwarp();
  };
  clear_acc();

  const uint32_t n_units = uint32_t(p.Q * p.S);
  const uint32_t Qu = uint32_t(p.Q);
  for (;;) {
    uint32_t u = 0;
    if (lane == 0) u = atomicAdd(p.next_unit, 1u);
    u = __shfl_sync(full, u, 0);
    if (u >= n_units) break;
    const int s = int(u / Qu);  // split-major: concurrent units share a slice of the index
    const int64_t q = u - uint32_t(s) * Qu;
    const int b0 = int((int64_t(s) * p.nblk) / p.S);
    const int b1 = int((int64_t(s + 1) * p.nblk) / p.S);
    const int qt0 = p.q_indptr[q];
    const int nterms = p.q_indptr[q + 1] - qt0;
    const int nchunks = nterms > 32 ? (nterms + 31) >> 5 : 1;  // a step = (G blocks, chunk of 32 query terms)
    const bool one_chunk = nchunks == 1;
    uint32_t* const floor_q = p.S > 1 ? p.floor_q + q : nullptr;
    SRFilter uf{};
    if (FILTERED) {
      const int fr = filter_row(p.filter, q);
      uf = SRFilter{p.filter.live, fr >= 0 ? p.filter.allow + int64_t(fr) * p.filter.ld_words : nullptr, p.filter.id_offset,
                    fr == FILTER_NONE ? 1 : 0};
    }
    auto candidate = [&](uint32_t nw, uint32_t old, uint32_t doc) {
      if constexpr (FILTERED) return sr_candidate(list, hist, st, floor_q, p.cap, p.k, nw, old, doc, uf);
      else return sr_candidate(list, hist, st, floor_q, p.cap, p.k, nw, old, doc);
    };

    // ---- candidate list of the unit: empty, or what the previous split of this query left behind
    {
      uint32_t n0 = 0;
      uint64_t thr0 = 0xFFFFFFFFull;  // every score-0 key is <= this
      if (s > 0 && p.unit_thr) {
        const int64_t prev = int64_t(s - 1) * p.Q + q;
        const uint64_t t = ld_acquire_u64(p.unit_thr + prev);
        if (t != 0) {  // that unit is complete (warp-uniform: every lane read the same word)
          n0 = uint32_t(__ldcg(p.counts + prev));
          thr0 = t;
          const uint64_t* src = p.cand + prev * p.cap;
          for (uint32_t i = lane; i < n0; i += 32) list[i] = ld_cg_u64(src + i);
          __syncwarp();
          if (lane == 0) p.counts[prev] = 0;  // its entries live on in this unit's list
        }
      }
      if (lane == 0) {
        st->n = n0;
        st->thr = thr0;
        st->min_sc = max(1u, key_hi(thr0));
      }
      __syncwarp();
    }
    uint32_t min_sc = st->min_sc;
    uint32_t floor_pref = 0;  // the query's global score floor, fetched when the loader entered its step
    uint32_t mxo = 0;         // OR of all sums (16-bit overflow check)

    // ---- loader state: lane t owns term t of the chunk being loaded
    const uint32_t* bp_row = nullptr;
    int64_t post_base = 0;
    uint32_t lo = 0, hi = 0, nxt = 0, my_w = 0;
    if (one_chunk && lane < nterms) {
      const int t = p.q_tok[qt0 + lane];
      const int w = p.q_cnt[qt0 + lane];
      if (t >= 0 && t < p.V && w > 0) {  // terms with a count <= 0 contribute nothing
        bp_row = p.blockptr + int64_t(t) * (p.nblk + 1);
        post_base = p.post_indptr[t];
        my_w = uint32_t(w);
        lo = bp_row[b0];
        hi = bp_row[min(b0 + G, b1)];
        nxt = bp_row[min(b0 + 2 * G, b1)];
      }
    }
    int lb, lc;          // step the loader is in: blocks [lb, min(lb + G, b1)), chunk lc
    int rL = 0, RL = 0;  // next row / number of rows of that step
    int rp = 0;          // rows of the lower lanes' terms (exclusive prefix)

    auto enter = [&]() {
      int cnt = 0;
      int64_t start = 0;
      uint32_t w = 0;
      if (one_chunk) {
        if (bp_row) {
          start = post_base + lo;
          cnt = int(hi - lo);
          w = my_w;
          lo = hi;
          hi = nxt;
          if (lb + 2 * G < b1) nxt = bp_row[min(lb + 3 * G, b1)];  // consumed two steps from now
        }
      } else {
        const int i = lc * 32 + lane;
        if (i < nterms) {
          const int t = p.q_tok[qt0 + i];
          const int wi = p.q_cnt[qt0 + i];
          if (t >= 0 && t < p.V && wi > 0) {
            const uint32_t* bp = p.blockptr + int64_t(t) * (p.nblk + 1);
            const uint32_t l2 = bp[lb], h2 = bp[min(lb + G, b1)];
            start = p.post_indptr[t] + l2;
            cnt = int(h2 - l2);
            w = uint32_t(wi);
          }
        }
      }
      if (floor_q) floor_pref = ld_relaxed_u32(floor_q);
      const int rows = (cnt + 31) >> 5;
      int incl = rows;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int t = __shfl_up_sync(full, incl, off);
        if (lane >= off) incl += t;
      }
      RL = __shfl_sync(full, incl, 31);
      rp = incl - rows;
      rL = 0;
      // posting j of the flattened row space (j = row * 32 + lane) of this lane's term sits at index A + j, for
      // j in [rp * 32, rp * 32 + cnt)
      const int64_t A = start - int64_t(rp) * 32;
      __syncwarp();  // the rows of the previous step have read the table
      tab[lane] = make_uint4(uint32_t(uint64_t(A)), uint32_t(uint64_t(A) >> 32), uint32_t(rp * 32 + cnt - 1), w);
      __syncwarp();
    };

    auto issue = [&](RowBatch<NB>& B) {
      while (rL >= RL) {  // next step with postings
        if (++lc == nchunks) {
          lc = 0;
          lb += G;
        }
        if (lb >= b1) {
          B.nb = 0;
          return;
        }
        enter();
      }
      B.d0 = lb * p.bd;
      {
        // long run: NB full rows of the term that owns row rL
        const uint32_t m = __ballot_sync(full, rp <= rL);  // lane 0 always votes; the highest voter owns the row
        const uint4 e = tab[31 - __clz(m)];
        if (((int(e.z) + 1) >> 5) - rL >= NBF) {  // warp-uniform
          const int64_t idx = int64_t((uint64_t(e.y) << 32) | uint64_t(e.x)) + (rL * 32 + lane);
          const int32_t* pd = p.post_doc + idx;
          const uint16_t* pi = p.post_imp + idx;
#pragma unroll
          for (int i = 0; i < NBF; ++i) {
            B.x[i] = uint32_t(__ldg(pd + i * 32));
            B.x[NBF + i] = uint32_t(__ldg(pi + i * 32));
          }
          B.w = e.w;
          B.nb = NBF;
          rL += NBF;
          return;
        }
      }
      B.w = 0;
      B.nb = min(NB, RL - rL);
#pragma unroll
      for (int i = 0; i < NB; ++i) {
        if (i < B.nb) {  // warp-uniform
          const int r = rL + i;
          const uint32_t m = __ballot_sync(full, rp <= r);
          const uint4 e = tab[31 - __clz(m)];
          const int j = r * 32 + lane;
          const int last = int(e.z);
          const int64_t idx = int64_t((uint64_t(e.y) << 32) | uint64_t(e.x)) + min(j, last);  // lanes past the end repeat the last posting
          B.x[i] = uint32_t(__ldg(p.post_doc + idx));
          B.x[NB + i] = uint32_t(__ldg(p.post_imp + idx));
          B.x[2 * NB + i] = j <= last ? e.w : 0u;
        }
      }
      rL += B.nb;
    };

    int cur_d0 = -1;
    bool dirty = false;
    auto consume = [&](const RowBatch<NB>& B) {
      if (B.d0 != cur_d0) {  // first batch of a new step (chunks of one step share d0)
        if (dirty) clear_acc();
        cur_d0 = B.d0;
        if (floor_pref > min_sc) {  // the floor only moves between steps: a listed document always met it
          min_sc = floor_pref;
          if (lane == 0) st->min_sc = min_sc;
          __syncwarp();
        }
      }
      dirty = true;
      AccT* const ab = acc - B.d0;  // indexed by document id
      if (B.w != 0) {
        // NBF full rows of one term: no two postings share a document, so the read-modify-writes are independent
        uint32_t old[NBF], nw[NBF];
#pragma unroll
        for (int i = 0; i < NBF; ++i) old[i] = uint32_t(ab[int(B.x[i])]);
        uint32_t hi_sc = 0;
#pragma unroll
        for (int i = 0; i < NBF; ++i) {
          nw[i] = old[i] + B.w * B.x[NBF + i];
          hi_sc = max(hi_sc, nw[i]);
          mxo |= nw[i];
        }
#pragma unroll
        for (int i = 0; i < NBF; ++i) ab[int(B.x[i])] = AccT(nw[i]);
        __syncwarp();
        if (__any_sync(full, hi_sc >= min_sc)) {
#pragma unroll
          for (int i = 0; i < NBF; ++i)
            if (__any_sync(full, nw[i] >= min_sc))
              min_sc = candidate(nw[i], old[i], B.x[i]);
        }
        return;
      }
#pragma unroll
      for (int i = 0; i < NB; ++i) {
        if (i < B.nb) {  // warp-uniform
          const uint32_t add = B.x[2 * NB + i] * B.x[NB + i];
          uint32_t old = 0, nw = 0;
          if (add != 0) {
            old = uint32_t(ab[int(B.x[i])]);
            nw = old + add;
            ab[int(B.x[i])] = AccT(nw);
            mxo |= nw;
          }
          __syncwarp();  // the next row may touch the same accumulators from other lanes
          if (__any_sync(full, nw >= min_sc))  // min_sc >= 1: idle lanes (nw == 0) never pass
            min_sc = candidate(nw, old, B.x[i]);
        }
      }
    };

    RowBatch<NB> A, B;
    lb = b0 - G;  // the first issue() advances to (b0, chunk 0)
    lc = nchunks - 1;
    issue(A);
    for (;;) {
      if (A.nb == 0) break;
      issue(B);  // in flight while A is accumulated
      consume(A);
      if (B.nb == 0) break;
      issue(A);
      consume(B);
    }
    if (dirty) clear_acc();
    if (sizeof(AccT) == 2 && __any_sync(full, mxo > 0xFFFFu) && lane == 0) atomicOr(p.overflow, 1u);
    // ---- unit result
    const uint32_t n = st->n;
    const int64_t ui = int64_t(s) * p.Q + q;
    uint64_t* dst = p.cand + ui * p.cap;
    for (uint32_t i = lane; i < n; i += 32) dst[i] = list[i];
    if (lane == 0) p.counts[ui] = int32_t(n);
    __syncwarp();
    if (p.unit_thr && lane == 0) st_release_u64(p.unit_thr + ui, st->thr);  // list + count are visible before this
    __syncwarp();
  }
}

}  // namespace lr
