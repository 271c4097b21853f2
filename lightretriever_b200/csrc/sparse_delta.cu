// sparse_delta.cu — exact impact scoring + top-k over a forward (document-major) segment: the append-only delta of an
// online searcher.
//
// K4 (sparse_score.cu) scores a token-major inverted index, which cannot grow in place.  Documents inserted while a
// searcher serves are stored document-major (doc_ptr / doc_tok / doc_imp, appended at the end) and scored here with
// K4's semantics: score(q, d) = sum over the postings of d of count_q(t) * impact_d(t) in 32-bit integers, so a token
// repeated in a document counts twice; only scores > 0 are returned; LR_SCORE_U32 keys; ties by ascending id.
//
// Work: a unit is (query, split of the filled documents); one warp per unit.  A CTA serves W units of ONE query and
// first stages that query's terms in shared memory as an open-addressing table keyed by token (a token listed twice
// sums its counts: the same integer as K4 adding both terms).  Each lane then scores one document at a time, walking
// its postings with one table probe each; documents beating the unit's running threshold key (and the filters) are
// appended to the warp's candidate list, cut to its exact top-k when full (warp_cut_topk).  The lists go through
// topk_merge_two_level, as K4's do.  Queries are processed in chunks so that the workspace stays bounded for offline
// batches.  The fill level *n_docs is read on the device: a call captured in a CUDA graph sees later appends.
#include "common.cuh"
#include "warp_topk.cuh"

namespace lr {

int topk_merge_two_level(const uint64_t* keys, const int32_t* counts, int L, int64_t Q, int64_t q_stride, int cap, int k,
                         int score_kind, int64_t id_offset, float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                         int64_t out_key_stride, void* scratch, size_t scratch_bytes, cudaStream_t st);
size_t topk_merge_scratch_bytes(int L, int64_t Q, int cap, int k);

constexpr int SF_TABLE_SLOTS = 2 * LR_QUERY_MAX_BAG;  // at most half full: every probe sequence ends at an empty slot
constexpr int SF_MAX_WARPS = 16;
constexpr int SF_UNROLL = 4;                          // postings per lane in flight
constexpr size_t SF_CHUNK_BYTES = size_t(64) << 20;   // candidate lists of one query chunk

struct SFParams {
  const int32_t* q_indptr;
  const int32_t* q_tok;
  const int32_t* q_cnt;
  int64_t q0, Qc;  // this launch scores queries [q0, q0 + Qc)
  const int64_t* doc_ptr;
  const int32_t* n_docs;
  const int32_t* doc_tok;
  const uint16_t* doc_imp;
  int64_t cap_docs, V;
  int k, cap, S, W;    // S = lists per query = CTAs per query x W warps
  uint64_t* cand;      // [S][Qc][cap]
  int32_t* counts;     // [S][Qc]
  DocFilter filter;
};

__device__ __forceinline__ uint32_t sf_hash(int32_t t, uint32_t mask) { return (uint32_t(t) * 0x9E3779B1u >> 7) & mask; }

__global__ void __launch_bounds__(SF_MAX_WARPS * 32, 1) sparse_fwd_kernel(const SFParams p) {
  extern __shared__ __align__(16) uint8_t sf_smem[];
  int32_t* tab_tok = reinterpret_cast<int32_t*>(sf_smem);
  int32_t* tab_cnt = tab_tok + SF_TABLE_SLOTS;
  const uint32_t full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* wbase = sf_smem + size_t(SF_TABLE_SLOTS) * 8 + size_t(warp) * (size_t(p.cap) * 8 + 1024);
  uint64_t* list = reinterpret_cast<uint64_t*>(wbase);
  uint32_t* hist = reinterpret_cast<uint32_t*>(list + p.cap);

  const int64_t ql = blockIdx.x / (p.S / p.W);
  const int s = int(blockIdx.x % (p.S / p.W)) * p.W + warp;
  const int64_t q = p.q0 + ql;
  int64_t nd = *p.n_docs;
  nd = nd < 0 ? 0 : (nd > p.cap_docs ? p.cap_docs : nd);

  // ---- the query's terms -> table (size: a power of two >= 2 x terms)
  const int qt0 = p.q_indptr[q];
  int nterms = p.q_indptr[q + 1] - qt0;
  nterms = nterms < 0 ? 0 : (nterms > LR_QUERY_MAX_BAG ? LR_QUERY_MAX_BAG : nterms);
  uint32_t slots = 32;
  while (slots < uint32_t(2 * nterms)) slots <<= 1;
  const uint32_t mask = slots - 1;
  for (uint32_t i = threadIdx.x; i < slots; i += blockDim.x) {
    tab_tok[i] = -1;
    tab_cnt[i] = 0;
  }
  __syncthreads();
  bool any = false;
  for (int i = threadIdx.x; i < nterms; i += blockDim.x) {
    const int32_t t = p.q_tok[qt0 + i];
    const int32_t w = p.q_cnt[qt0 + i];
    if (t < 0 || t >= p.V || w <= 0) continue;  // terms with a count <= 0 contribute nothing (as in K4)
    any = true;
    for (uint32_t h = sf_hash(t, mask);; h = (h + 1) & mask) {
      const int32_t old = atomicCAS(&tab_tok[h], -1, t);
      if (old == -1 || old == t) {
        atomicAdd(&tab_cnt[h], w);
        break;
      }
    }
  }
  any = __syncthreads_or(any);

  // ---- this warp's documents [d0, d1)
  uint32_t n = 0;                // entries in `list` (warp-uniform)
  uint64_t thr = 0xFFFFFFFFull;  // candidates need key > thr; every score-0 key is <= this
  if (any) {
    const int64_t d0 = nd * s / p.S, d1 = nd * (s + 1) / p.S;
    const int f_row = p.filter.on ? filter_row(p.filter, q) : FILTER_ALL;
    const uint32_t lt = lanemask_lt();
    for (int64_t base = d0; base < d1; base += 32) {
      const int64_t d = base + lane;
      uint32_t sc = 0;
      if (d < d1) {
        const int64_t e = p.doc_ptr[d + 1];
        int64_t j = p.doc_ptr[d];
        for (; j + SF_UNROLL <= e; j += SF_UNROLL) {
          int32_t t[SF_UNROLL], m[SF_UNROLL];
#pragma unroll
          for (int u = 0; u < SF_UNROLL; ++u) {
            t[u] = __ldg(p.doc_tok + j + u);
            m[u] = int32_t(__ldg(p.doc_imp + j + u));
          }
#pragma unroll
          for (int u = 0; u < SF_UNROLL; ++u) {
            for (uint32_t h = sf_hash(t[u], mask);; h = (h + 1) & mask) {
              const int32_t tt = tab_tok[h];
              if (tt == t[u]) {
                sc += uint32_t(tab_cnt[h] * m[u]);
                break;
              }
              if (tt == -1) break;
            }
          }
        }
        for (; j < e; ++j) {
          const int32_t t = __ldg(p.doc_tok + j);
          const int32_t m = int32_t(__ldg(p.doc_imp + j));
          for (uint32_t h = sf_hash(t, mask);; h = (h + 1) & mask) {
            const int32_t tt = tab_tok[h];
            if (tt == t) {
              sc += uint32_t(tab_cnt[h] * m);
              break;
            }
            if (tt == -1) break;
          }
        }
      }
      const uint64_t key = make_key(sc, uint32_t(d));
      bool pass = d < d1 && key > thr;  // key > thr implies sc > 0
      if (pass && p.filter.on) pass = filter_allows(p.filter, f_row, d);
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
          pass = pass && key > thr;
        }
        pm = __ballot_sync(full, pass);
      }
    }
  }
  // ---- unit result
  uint64_t* dst = p.cand + (int64_t(s) * p.Qc + ql) * p.cap;
  __syncwarp();
  for (uint32_t i = lane; i < n; i += 32) dst[i] = list[i];
  if (lane == 0) p.counts[int64_t(s) * p.Qc + ql] = int32_t(n);
}

struct SFPlan {
  int cap, W, G, S;  // list capacity, warps per CTA, CTAs per query, lists per query
  int64_t Qc;        // queries per chunk
  size_t smem, off_cand, off_merge, merge_bytes, total_bytes;
};

static size_t sf_align(size_t x) { return (x + 255) / 256 * 256; }

static SFPlan sf_plan(int64_t Q, int64_t cap_docs, int k) {
  SFPlan pl{};
  const int cap = k + (k / 2 > 156 ? k / 2 : 156);  // K4's list capacity (k = 100 -> 256)
  pl.cap = (cap + 31) / 32 * 32;
  const size_t warp_bytes = size_t(pl.cap) * 8 + 1024;
  const size_t room = size_t(227) * 1024 - 1024 - size_t(SF_TABLE_SLOTS) * 8;
  int W = int(room / warp_bytes);
  pl.W = W > SF_MAX_WARPS ? SF_MAX_WARPS : (W < 1 ? 1 : W);
  pl.smem = size_t(SF_TABLE_SLOTS) * 8 + size_t(pl.W) * warp_bytes;
  // CTAs per query: two per SM over the batch, but no more than leave each warp 32 documents of a full segment
  const int64_t G = sm_count();
  auto ctas = [&](int64_t Qc) {
    int64_t g = (2 * G + Qc - 1) / Qc;
    const int64_t by_docs = (cap_docs + 32 * pl.W - 1) / (32 * pl.W);
    if (g > by_docs) g = by_docs;
    if (g > 64) g = 64;
    return int(g < 1 ? 1 : g);
  };
  int64_t Qc = Q < 4096 ? Q : 4096;
  while (Qc > 1 && size_t(ctas(Qc)) * pl.W * size_t(Qc) * pl.cap * 8 > SF_CHUNK_BYTES) Qc = (Qc + 1) / 2;
  pl.Qc = Qc;
  pl.G = ctas(Qc);
  pl.S = pl.G * pl.W;
  const int64_t last = Q % Qc;
  pl.off_cand = sf_align(size_t(pl.S) * Qc * 4);
  pl.off_merge = sf_align(pl.off_cand + size_t(pl.S) * Qc * pl.cap * 8);
  size_t mb = topk_merge_scratch_bytes(pl.S, Qc, pl.cap, k);
  if (last) {
    const size_t mb2 = topk_merge_scratch_bytes(pl.S, last, pl.cap, k);
    mb = mb2 > mb ? mb2 : mb;
  }
  pl.merge_bytes = mb;
  pl.total_bytes = sf_align(pl.off_merge + mb);
  return pl;
}

}  // namespace lr

using namespace lr;

extern "C" size_t lr_sparse_fwd_workspace_bytes(int64_t Q, int64_t cap_docs, int k) {
  if (Q < 1 || cap_docs < 0 || k < 1 || k > 1024) return 0;
  return sf_plan(Q, cap_docs, k).total_bytes;
}

extern "C" int lr_sparse_fwd_score_topk(const int32_t* q_indptr, const int32_t* q_tok, const int32_t* q_cnt, int64_t Q,
                                        const int64_t* doc_ptr, const int32_t* n_docs, const int32_t* doc_tok,
                                        const uint16_t* doc_imp, int64_t cap_docs, int64_t V, int64_t id_offset, int k,
                                        float* out_scores, int64_t* out_ids, uint64_t* out_keys, const uint32_t* live,
                                        const uint32_t* allow, int64_t ld_words, int n_filters, const int32_t* q_filter,
                                        void* workspace, size_t ws_bytes, void* stream) {
  LR_CHECK_ARG(q_indptr && q_tok && q_cnt && doc_ptr && n_docs && doc_tok && doc_imp, "sparse_fwd: null pointer");
  LR_CHECK_ARG(Q >= 1 && V >= 1, "sparse_fwd: Q and V must be >= 1");
  LR_CHECK_ARG(cap_docs >= 0 && cap_docs < (int64_t(1) << 31), "sparse_fwd: cap_docs (%lld) must be in [0, 2^31)",
               (long long)cap_docs);
  LR_CHECK_ARG(k >= 1 && k <= 1024, "sparse_fwd: k (%d) must be in [1, 1024]", k);
  LR_CHECK_ARG(id_offset >= 0 && id_offset + cap_docs <= (int64_t(1) << 32) - 2,
               "sparse_fwd: id_offset + cap_docs must stay below 2^32");
  LR_CHECK_ARG(out_scores || out_ids || out_keys, "sparse_fwd: no output requested");
  DocFilter flt;
  if (int frc = make_doc_filter(live, allow, ld_words, n_filters, q_filter, id_offset, cap_docs, flt)) return frc;
  const SFPlan pl = sf_plan(Q, cap_docs, k);
  if (!workspace || ws_bytes < pl.total_bytes || (uintptr_t(workspace) & 255)) {
    set_error("sparse_fwd: workspace too small or misaligned (%zu given, %zu needed)", ws_bytes, pl.total_bytes);
    return LR_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  SFParams p{};
  p.q_indptr = q_indptr; p.q_tok = q_tok; p.q_cnt = q_cnt;
  p.doc_ptr = doc_ptr; p.n_docs = n_docs; p.doc_tok = doc_tok; p.doc_imp = doc_imp;
  p.cap_docs = cap_docs; p.V = V; p.k = k; p.cap = pl.cap; p.S = pl.S; p.W = pl.W;
  p.counts = reinterpret_cast<int32_t*>(ws);
  p.cand = reinterpret_cast<uint64_t*>(ws + pl.off_cand);
  p.filter = flt;
  int rc = ensure_dyn_smem(reinterpret_cast<const void*>(sparse_fwd_kernel), 227 * 1024);
  if (rc) return rc;
  for (int64_t q0 = 0; q0 < Q; q0 += pl.Qc) {
    const int64_t qc = Q - q0 < pl.Qc ? Q - q0 : pl.Qc;
    p.q0 = q0;
    p.Qc = qc;
    sparse_fwd_kernel<<<unsigned(qc * pl.G), pl.W * 32, pl.smem, st>>>(p);
    LR_LAUNCH_CHECK();
    rc = topk_merge_two_level(p.cand, p.counts, pl.S, qc, qc, pl.cap, k, LR_SCORE_U32, id_offset,
                              out_scores ? out_scores + q0 * k : nullptr, out_ids ? out_ids + q0 * k : nullptr,
                              out_keys ? out_keys + q0 * k : nullptr, k, ws + pl.off_merge, pl.merge_bytes, st);
    if (rc) return rc;
  }
  return LR_OK;
}
