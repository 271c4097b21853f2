// flatip_topk.cu — K2: exact flat inner-product top-k on B200 (host side: plan, tensor maps, launches).
//
// Replaces faiss.IndexFlatIP.search as called by FaissIndex.search
// (reference retriever/faiss_index.py:27-40) plus the per-chunk heap merge
// (retriever/hybrid_search.py:182-205).  The kernel is umma_gemm_kernel<EPI_TOPK> in umma_gemm.cuh:
// rows = queries, columns = documents, the epilogue keeps per-(split, query) candidate lists which
// topk_merge reduces to the final sorted top-k.
//
// Large searches run in two phases.  Phase A scores a short corpus prefix and seeds every query's running
// threshold with its k-th best score there (any k documents give a valid lower bound of the final k-th score);
// phase B scores the rest with warm thresholds, so almost nothing is appended to the candidate lists and the
// list compactions that would stall the MMA pipe (and desynchronise the CTAs that share corpus tiles in L2)
// all but disappear.  The prefix's own top-k joins the final merge as one more candidate list.
#include "umma_gemm.cuh"

namespace lr {

int topk_merge_two_level(const uint64_t* keys, const int32_t* counts, int L, int64_t Q, int64_t q_stride, int cap, int k,
                         int score_kind, int64_t id_offset, float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                         int64_t out_key_stride, void* scratch, size_t scratch_bytes, cudaStream_t st);
size_t topk_merge_scratch_bytes(int L, int64_t Q, int cap, int k);

struct PassPlan {
  int tile_begin, tile_end, splits, units, grid, rounds;
  int sched, band_size, n_bands;  // sched 1: fixed teams per band (band_size groups per full band)
};
constexpr int MAX_MID = 6;
struct FlatipPlan {
  int cl, pair, m_groups, m_tiles, n_tiles, band_size, n_bands, cap, n_clusters;
  int64_t q_pad;
  PassPlan main, prefix;  // prefix.units == 0 -> single phase
  // Epilogue-bound searches (short rows, d_used <= 1024) refresh the thresholds more than once: passes over geometrically
  // growing tile ranges between the prefix and the main pass, each followed by a merge that re-seeds every query's
  // threshold with its k-th best score so far.
  int n_mid;
  PassPlan mid[MAX_MID];
  int wide;  // two epilogue warp sets (umma_gemm.cuh WIDE): every split owns TWO candidate lists
  int lmul;  // candidate lists per split (1 or 2)
  int max_lists;  // lists of the widest pass + 1 (the carried top-k)
  size_t off_gthr, off_counts, off_cand, off_pcounts, off_pcand, off_carry, off_teamctr, off_merge, merge_bytes, total_bytes;
};

// Team schedule of the main pass: bands of g row groups; inside a band the clusters form floor(nc / g) fixed teams, each
// walking its own splits with one cluster per row group (so a B tile is fetched once per team and the members are kept
// within a small window by a progress counter).  Picks g and the split count for high cluster utilisation, few corpus
// passes and an L2-resident A band (<= 40 MB = 20 groups of 2 x 128 rows x 8 KB).
static bool plan_teams(int m_groups, int nc, int n_tiles_pass, int64_t s_cap, PassPlan& pp) {
  double best = -1.0;
  int best_g = 0, best_s = 0;
  const int g_hi = m_groups < 20 ? m_groups : 20, g_lo = m_groups < 4 ? m_groups : 4;
  for (int g = g_lo; g <= g_hi; ++g) {
    if (g > nc) break;
    const int q = m_groups / g, r = m_groups % g;
    const int n_main = nc / g, n_rem = r ? nc / r : 0;
    for (int mult = 1; mult <= 64; ++mult) {
      const int S = n_main * mult;
      if (S > s_cap || S > n_tiles_pass || S > 96) break;
      const int64_t time = int64_t(q) * ((S + n_main - 1) / n_main) + (r ? (S + n_rem - 1) / n_rem : 0);
      const double util = double(m_groups) * S / (double(nc) * double(time));
      const int passes = q + (r ? 1 : 0);
      const int64_t tiles_per_split = n_tiles_pass / S;
      double score = util - 0.012 * passes - (tiles_per_split < 64 ? 0.05 : 0.0) - 0.0002 * S;
      if (score > best) {
        best = score;
        best_g = g;
        best_s = S;
      }
    }
  }
  if (best_g == 0) return false;
  pp.sched = 1;
  pp.band_size = best_g;
  pp.n_bands = (m_groups + best_g - 1) / best_g;
  pp.splits = best_s;
  pp.units = m_groups * best_s;
  pp.grid = nc;
  const int q = m_groups / best_g, r = m_groups % best_g;
  const int n_main = nc / best_g, n_rem = r ? nc / r : 0;
  pp.rounds = q * ((best_s + n_main - 1) / n_main) + (r ? (best_s + n_rem - 1) / n_rem : 0);
  return true;
}

// corpus splits of one pass: minimise rounds * tiles-per-unit; accept a larger split count only for a >0.5% gain
static PassPlan plan_pass(int m_groups, int n_clusters, int tile_begin, int tile_end, int64_t s_cap, int forced) {
  PassPlan pp{};
  pp.tile_begin = tile_begin;
  pp.tile_end = tile_end;
  const int nt = tile_end - tile_begin;
  int64_t s_max = int64_t(4) * n_clusters;
  if (s_max > s_cap) s_max = s_cap;
  if (s_max > nt) s_max = nt;
  if (s_max < 1) s_max = 1;
  double best = 1e300;
  int best_s = 1;
  for (int64_t s = 1; s <= s_max; ++s) {
    const int64_t units = int64_t(m_groups) * s;
    const int64_t rounds = (units + n_clusters - 1) / n_clusters;
    const int64_t tiles = (nt + s - 1) / s;
    const double cost = double(rounds) * double(tiles + 1);  // +1: per-unit start-up
    if (cost < best * (1.0 - 0.005)) {
      best = cost;
      best_s = int(s);
    }
  }
  if (forced > 0 && forced <= nt) best_s = forced;
  pp.splits = best_s;
  pp.units = m_groups * pp.splits;
  int clusters = pp.units < n_clusters ? pp.units : n_clusters;
  if (clusters < 1) clusters = 1;
  pp.grid = clusters;  // in clusters; multiplied by cl at launch
  pp.rounds = (pp.units + clusters - 1) / clusters;
  return pp;
}

static FlatipPlan make_plan_uncached(int64_t Q, int64_t N, int k, int64_t d_used, int shards) {
  FlatipPlan pl{};
  const Knobs& kn = knobs();
  // Candidate-list capacity.  The running threshold of a row only rises when its list is cut back to the top-k, so
  // between two cuts exactly cap-k entries are admitted and the number of documents consumed grows by cap/k per cut;
  // measured on B200 (profiles/): 2k..2.5k beats both smaller and larger lists.
  int cap = 2 * k > k + 64 ? 2 * k : k + 64;
  if (k <= 128 && cap < 256) cap = 256;
  pl.cap = (cap + 63) / 64 * 64;
  // Kernel variant.  Small batches: cluster of 2 with multicast B.  Long lists (k > 352: a list no longer fits the
  // 6 KB/warp staging area) run as a cta_group::2 pair with the BIGLIST layout (4 stages of 32 KB + 22 KB/warp of list
  // staging): there the epilogue is the limiter — measured at k=1000, 8.8M docs: 841 ms (multicast) -> 660 ms (pair +
  // BIGLIST + 256k-document prefix).  Large batches on the team schedule also run as pairs: once the corpus tiles stay
  // L2-resident the halved shared-memory traffic of cta_group::2 is what the power cap rewards (same box, 8.8M x 4096,
  // k=100: 585 ms multicast vs 537 ms pair; profiles/k2_ab_same_box_r1.jsonl).
  int mode = kn.flatip_cluster;
  const bool long_lists = pl.cap > LIST_STAGE_ENTRIES;
  const bool team_sched = (Q + 2 * BM - 1) / (2 * BM) >= 8;
  if (mode == 0 && Q > BM && (long_lists || team_sched)) mode = 3;
  const GemmGeometry geo = plan_geometry(Q, 32, mode);  // bands of up to 32 query tiles
  pl.cl = geo.cl; pl.pair = geo.pair; pl.m_groups = geo.m_groups; pl.m_tiles = geo.m_tiles;
  pl.band_size = geo.band_size; pl.n_bands = geo.n_bands; pl.n_clusters = geo.n_clusters;
  pl.n_tiles = int((N + BN - 1) / BN);
  pl.q_pad = int64_t(pl.m_tiles) * BM;
  // Short rows (MRL prefixes): a 128x256 tile needs d_used/16 MMAs of 128 cycles but ~4-5k cycles of one epilogue warp
  // per TMEM lane quarter, so below ~768 columns the epilogue sets the pace: run two epilogue sets on alternate tiles.
  pl.wide = d_used <= 768 && Q > BM && !long_lists;
  pl.lmul = pl.wide ? 2 : 1;
  const int64_t list_bytes = pl.q_pad * int64_t(pl.cap) * 8 * pl.lmul;
  const int64_t s_cap = (int64_t(12) << 30) / (list_bytes > 0 ? list_bytes : 1);

  // Phase A (warm start) when the search is compute-bound and long enough to amortise it.  Measured on the 1.1M x 4096
  // shard shape (profiles/k2_schedule_sweeps_r1.md): a 32768-document prefix brings the main pass within 2% of a run
  // with perfect thresholds; 4k..8k-document prefixes do not pay for themselves.
  int prefix_tiles = 0, pt_global = 0;
  int prefix_splits_forced = 0;
  const int want = kn.flatip_prefix_docs;
  if (want != 0) {
    // default prefix: 256 documents per requested result, at least 32768, at most 1/16 of the corpus.  (Long lists,
    // k > 352: a 32768-document prefix with refresh passes forced on — a short warm start plus threshold-refresh passes
    // instead of one cold 256k-document pass — measured 577 -> 567 ms at 8.8M and 83.7 -> 80.6 ms at 1.1M for k = 1000 on
    // the same box; it stays an option until the full GPU suite has run with it.)
    const int64_t default_docs = int64_t(256) * k > 32768 ? int64_t(256) * k : 32768;
    int64_t docs = want > 0 ? want : default_docs;
    if (docs < 4 * int64_t(k)) docs = 4 * int64_t(k);
    int pt = int((docs + BN - 1) / BN);
    if (want < 0 && pt > pl.n_tiles / 16) pt = pl.n_tiles / 16;
    const bool big_enough = want > 0 || (pl.m_groups >= 4 && pt >= 128 && pl.n_tiles >= 32 * 128);
    // Row-sharded search (lr_flatip_topk_begin / _finish): this shard scores 1/shards of the warm-start prefix and the
    // caller exchanges the per-shard prefix top-k, so every shard starts the main pass with the k-th best score of the
    // whole prefix — the thresholds of the unsharded search at 1/shards of its warm-start cost per GPU.
    pt_global = pt;
    if (shards > 1) {
      pt = (pt + shards - 1) / shards;
      const int min_pt = int((2 * int64_t(k) + BN - 1) / BN);
      if (pt < min_pt) pt = min_pt;
    }
    if (big_enough && pt < pl.n_tiles) prefix_tiles = pt;
    // Small query batches (online serving, HBM-bound): a prefix of one tile per cluster, every cluster scoring a
    // different tile, costs one tile time and removes the cold-start cuts, which otherwise pile up in the one or two
    // epilogue warps that own the few valid query rows.
    if (want < 0 && pl.m_groups < 4 && Q >= 4) {  // one query: measured 1.37 ms single-phase vs 1.47 ms with the pass
      const int s0 = geo.n_clusters / pl.m_groups;
      if (s0 >= 8 && pl.n_tiles >= 8 * s0 && 4 * int64_t(k) <= int64_t(s0) * BN) {
        prefix_tiles = s0;
        prefix_splits_forced = s0;
        if (pl.cap < BN + 64) pl.cap = BN + 64;  // a one-tile unit never has to cut its list
      }
    }
  }
  if (prefix_tiles > 0)
    pl.prefix = plan_pass(pl.m_groups, geo.n_clusters, 0, prefix_tiles, s_cap, prefix_splits_forced);
  // Threshold refreshes for epilogue-bound searches: with d_used <= 1024 a tile's MMAs are shorter than its epilogue,
  // so every candidate appended under a stale threshold costs wall time.  Measured at 10k x 1.1M (profiles/): the lists
  // of a single main pass take k*N/prefix = 3.4k candidates per query; ranges growing 4x per pass bring that below 1k.
  int main_begin = prefix_tiles;
  pl.n_mid = 0;
  // (by default only with the default prefix size; the refresh knob set to 1 forces it for any prefix, e.g. for long lists)
  const int refresh = kn.flatip_refresh >= 0 ? kn.flatip_refresh : (d_used <= 1024 ? 1 : 0);
  const bool default_prefix = pt_global == int((int64_t(256) * k > 32768 ? int64_t(256) * k : 32768) / BN);
  if (refresh && pt_global >= 128 && prefix_tiles > 0 && prefix_splits_forced == 0 &&
      (default_prefix || kn.flatip_refresh > 0)) {
    constexpr int growth = 4;
    // ranges end at growth^i times the WHOLE prefix (a shard's thresholds start from the exchanged k-th best of it)
    int64_t end = int64_t(pt_global) * growth;
    while (pl.n_mid < MAX_MID && end + (end - main_begin) < pl.n_tiles) {
      pl.mid[pl.n_mid] = plan_pass(pl.m_groups, geo.n_clusters, main_begin, int(end), s_cap, 0);
      pl.mid[pl.n_mid].band_size = pl.band_size;
      pl.mid[pl.n_mid].n_bands = pl.n_bands;
      ++pl.n_mid;
      main_begin = int(end);
      end *= growth;
    }
  }
  pl.main = plan_pass(pl.m_groups, geo.n_clusters, main_begin, pl.n_tiles, s_cap, 0);
  pl.main.band_size = pl.band_size;
  pl.main.n_bands = pl.n_bands;
  pl.prefix.band_size = pl.band_size;
  pl.prefix.n_bands = pl.n_bands;
  // Large batches: fixed teams (see plan_teams).
  if (pl.cl == 2 && pl.m_groups >= 8) {
    PassPlan tp = pl.main;
    if (plan_teams(pl.m_groups, geo.n_clusters, pl.n_tiles - main_begin, s_cap, tp)) pl.main = tp;
  }

  auto align = [](size_t x) { return (x + 255) / 256 * 256; };
  int main_lists = pl.main.splits;
  for (int i = 0; i < pl.n_mid; ++i) main_lists = pl.mid[i].splits > main_lists ? pl.mid[i].splits : main_lists;
  main_lists = main_lists * pl.lmul + (prefix_tiles > 0 ? 1 : 0);  // + the carried top-k of the earlier passes
  pl.max_lists = main_lists;
  pl.off_gthr = 0;
  pl.off_counts = align(size_t(pl.q_pad) * 4);
  pl.off_cand = align(pl.off_counts + size_t(main_lists) * pl.q_pad * 4);
  pl.off_pcounts = align(pl.off_cand + size_t(main_lists) * pl.q_pad * pl.cap * 8);
  pl.off_pcand = align(pl.off_pcounts + size_t(pl.prefix.splits) * pl.lmul * pl.q_pad * 4);
  pl.off_carry = align(pl.off_pcand + size_t(pl.prefix.splits) * pl.lmul * pl.q_pad * pl.cap * 8);
  pl.off_teamctr = align(pl.off_carry + (prefix_tiles > 0 ? size_t(pl.q_pad) * pl.cap * 8 : 0));
  pl.off_merge = align(pl.off_teamctr + size_t(pl.main.n_bands) * size_t(pl.n_clusters) * 4 + 256);
  // scratch of the two-level merges (few queries, many lists: the online shapes)
  pl.merge_bytes = topk_merge_scratch_bytes(main_lists, Q, pl.cap, k);
  const size_t pm = topk_merge_scratch_bytes(pl.prefix.splits * pl.lmul, Q, pl.cap, k);
  if (pm > pl.merge_bytes) pl.merge_bytes = pm;
  pl.total_bytes = align(pl.off_merge + pl.merge_bytes);
  return pl;
}

// The planner loops (plan_pass: up to 4 x clusters split counts; plan_teams: band widths x multiples) run once per search
// shape: the online path repeats the same (Q, N, k, d_used) every request.  Per-thread cache, dropped on lr_reload_env().
static const FlatipPlan& make_plan(int64_t Q, int64_t N, int k, int64_t d_used, int shards = 1) {
  struct Entry {
    int64_t Q, N, d_used;
    int k, sms, shards;
    FlatipPlan pl;
  };
  constexpr int kEntries = 16;
  static thread_local Entry cache[kEntries];
  static thread_local int n_cached = 0, next_slot = 0;
  static thread_local unsigned epoch = 0;
  if (epoch != env_epoch()) {
    n_cached = next_slot = 0;
    epoch = env_epoch();
  }
  const int sms = sm_count();
  for (int i = 0; i < n_cached; ++i) {
    const Entry& e = cache[i];
    if (e.Q == Q && e.N == N && e.k == k && e.d_used == d_used && e.sms == sms && e.shards == shards) return e.pl;
  }
  Entry& e = cache[next_slot];
  next_slot = (next_slot + 1) % kEntries;
  if (n_cached < kEntries) ++n_cached;
  e.Q = Q; e.N = N; e.k = k; e.d_used = d_used; e.sms = sms; e.shards = shards;
  e.pl = make_plan_uncached(Q, N, k, d_used, shards);
  return e.pl;
}

static thread_local FlatipPlan g_last_plan{};

static int check_flatip_args(const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q, int64_t N,
                             int64_t d_used) {
  LR_CHECK_ARG(q && corpus, "flatip: null q or corpus");
  LR_CHECK_ARG(Q >= 1 && N >= 1, "flatip: Q (%lld) and N (%lld) must be >= 1", (long long)Q, (long long)N);
  LR_CHECK_ARG(N < (int64_t(1) << 31) - BN, "flatip: N (%lld) must be < 2^31 per shard", (long long)N);
  LR_CHECK_ARG(Q < (int64_t(1) << 31) - BM, "flatip: Q (%lld) too large", (long long)Q);
  LR_CHECK_ARG(d_used >= 8 && d_used % 8 == 0, "flatip: d_used (%lld) must be a positive multiple of 8", (long long)d_used);
  LR_CHECK_ARG(ldq >= d_used && ldc >= d_used, "flatip: row pitch (ldq=%lld, ldc=%lld) < d_used (%lld)",
               (long long)ldq, (long long)ldc, (long long)d_used);
  LR_CHECK_ARG((ldq * 2) % 16 == 0 && (ldc * 2) % 16 == 0, "flatip: row pitch must be a multiple of 16 bytes");
  LR_CHECK_ARG((uintptr_t(q) & 15) == 0 && (uintptr_t(corpus) & 15) == 0, "flatip: q/corpus must be 16-byte aligned");
  return LR_OK;
}

static void fill_params(GemmParams& prm, const FlatipPlan& pl, const PassPlan& pp, int64_t Q, int64_t N, int64_t d_used) {
  prm.rows = Q; prm.cols = N; prm.row_pad = pl.q_pad;
  prm.kblocks = int((d_used + BK - 1) / BK);
  prm.m_tiles = pl.m_tiles; prm.m_groups = pl.m_groups;
  prm.tile_begin = pp.tile_begin; prm.n_tiles = pp.tile_end; prm.splits = pp.splits;
  prm.band_size = pp.band_size ? pp.band_size : pl.band_size;  // plan_pass leaves the band layout to the geometry
  prm.n_bands = pp.band_size ? pp.n_bands : pl.n_bands; prm.units = pp.units;
  prm.sched = pp.sched;
  // The window is worth one full-width tile of operand traffic (64 k-blocks): with MRL prefixes (2..16 k-blocks per tile)
  // a one-tile window would make the team counter round trip — not the MMA — the pace of the kernel.
  prm.team_window = prm.kblocks >= 64 ? 1 : (64 + prm.kblocks - 1) / prm.kblocks;
}

template <int EPI>
static int launch_pass(const FlatipPlan& pl, const PassPlan& pp, const CUtensorMap& tmA, const CUtensorMap& tmB,
                       const GemmParams& prm, cudaStream_t st) {
  // Long candidate lists (k > 352): the BIGLIST layout gives the epilogue warps a larger list-staging area.  For a pair
  // it is free (4 of 6 stages of 32 KB keep the prefetch depth); for the multicast cluster it costs one of four 48 KB
  // stages, which only pays in short units (k=1000: 129 -> 107 ms at 390 tiles per unit, 810 -> 833 ms at 1427).
  const int tiles_per_unit = (pp.tile_end - pp.tile_begin + pp.splits - 1) / pp.splits;
  const bool big = EPI == EPI_TOPK && pl.cap > LIST_STAGE_ENTRIES && (pl.pair || tiles_per_unit < 1000);
  if (big) {
    if (pl.pair) return launch_umma_gemm<EPI_TOPK, 2, true, true>(tmA, tmB, prm, pp.grid * 2, st);
    return pl.cl == 2 ? launch_umma_gemm<EPI_TOPK, 2, false, true>(tmA, tmB, prm, pp.grid * 2, st)
                      : launch_umma_gemm<EPI_TOPK, 1, false, true>(tmA, tmB, prm, pp.grid, st);
  }
  if (EPI == EPI_TOPK && pl.wide) {
    if (pl.pair) return launch_umma_gemm<EPI_TOPK, 2, true, false, true>(tmA, tmB, prm, pp.grid * 2, st);
    return pl.cl == 2 ? launch_umma_gemm<EPI_TOPK, 2, false, false, true>(tmA, tmB, prm, pp.grid * 2, st)
                      : launch_umma_gemm<EPI_TOPK, 1, false, false, true>(tmA, tmB, prm, pp.grid, st);
  }
  if (pl.pair) return launch_umma_gemm<EPI, 2, true>(tmA, tmB, prm, pp.grid * 2, st);
  return pl.cl == 2 ? launch_umma_gemm<EPI, 2>(tmA, tmB, prm, pp.grid * 2, st)
                    : launch_umma_gemm<EPI, 1>(tmA, tmB, prm, pp.grid, st);
}

// Carries the merged top-k of the passes so far into the next pass: copies the k keys of every query into that pass's
// extra candidate list (counts = k), and seeds gthr[q] with the score key of the k-th best (0 when fewer than k
// documents have been seen — any k documents give a valid lower bound of the final k-th score).
__global__ void carry_topk_kernel(const uint64_t* __restrict__ merged, int64_t key_stride, int k, int64_t q_pad,
                                  int64_t Q, uint64_t* __restrict__ dst, uint32_t* __restrict__ gthr,
                                  int32_t* __restrict__ counts, const uint64_t* __restrict__ seed) {
  const int64_t q = blockIdx.x;
  if (q >= q_pad) return;
  __shared__ uint32_t s_g;
  __shared__ int s_n;
  if (threadIdx.x == 0) {
    uint32_t g = 0;
    if (q < Q) {
      const uint64_t kth = merged[q * key_stride + (k - 1)];
      if (kth != 0ull) g = key_hi(kth);
      if (seed) {  // [Q, k] sorted keys of the union of every shard's prefix: its k-th best bounds the global k-th score
        const uint64_t sk = seed[q * int64_t(k) + (k - 1)];
        if (sk != 0ull && key_hi(sk) > g) g = key_hi(sk);
      }
    }
    gthr[q] = g;
    s_g = g;
    s_n = 0;
  }
  __syncthreads();
  if (q < Q) {
    // the list is sorted: the entries that still reach the (possibly seeded) threshold are a leading run
    const uint32_t g = s_g;
    int n = 0;
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
      const uint64_t key = merged[q * key_stride + i];
      dst[q * key_stride + i] = key;
      n += (key != 0ull && key_hi(key) >= g) ? 1 : 0;
    }
    if (n) atomicAdd(&s_n, n);
  }
  __syncthreads();
  if (threadIdx.x == 0) counts[q] = q < Q ? s_n : 0;
}

// gthr[q] = max(gthr[q], score key of seed[q][k-1]) for a sharded search whose local plan has no warm-start pass
__global__ void seed_thresholds_kernel(const uint64_t* __restrict__ seed, int k, int64_t Q, uint32_t* __restrict__ gthr) {
  const int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  const uint64_t sk = seed[q * int64_t(k) + (k - 1)];
  if (sk != 0ull && key_hi(sk) > gthr[q]) gthr[q] = key_hi(sk);
}

}  // namespace lr

using namespace lr;

extern "C" size_t lr_flatip_workspace_bytes_for(int64_t Q, int64_t N, int k, int64_t d_used) {
  if (Q < 1 || N < 1 || k < 1 || d_used < 1) return 0;
  return make_plan(Q, N, k, d_used).total_bytes;
}

extern "C" size_t lr_flatip_workspace_bytes(int64_t Q, int64_t N, int k) {
  if (Q < 1 || N < 1 || k < 1) return 0;
  // the plan depends on d_used only through its regime: short rows (two lists per split, refresh passes) or not
  const size_t a = make_plan(Q, N, k, 4096).total_bytes, b = make_plan(Q, N, k, 64).total_bytes;
  return a > b ? a : b;
}

// Plan of a (Q, N, k) search without running it (no device needed beyond the SM count): for tests and capacity planning.
// out[0]=cluster size (1|2) out[1]=pair (0|1) out[2]=m_tiles out[3]=n_tiles out[4]=cap out[5]=prefix tile_end
// out[6]=prefix splits out[7]=prefix units out[8]=main tile_begin out[9]=main splits out[10]=main units
// out[11]=main grid (CTAs) out[12]=band (row tiles) out[13]=workspace bytes out[14]=main rounds out[15]=n_clusters
extern "C" int lr_flatip_plan(int64_t Q, int64_t N, int k, int64_t* out16) {
  LR_CHECK_ARG(out16 && Q >= 1 && N >= 1 && k >= 1 && k <= 2048, "flatip_plan: bad arguments");
  const FlatipPlan pl = make_plan(Q, N, k, 4096);
  out16[0] = pl.cl; out16[1] = pl.pair; out16[2] = pl.m_tiles; out16[3] = pl.n_tiles; out16[4] = pl.cap;
  out16[5] = pl.prefix.tile_end; out16[6] = pl.prefix.splits; out16[7] = pl.prefix.units;
  out16[8] = pl.main.tile_begin; out16[9] = pl.main.splits; out16[10] = pl.main.units;
  out16[11] = int64_t(pl.main.grid) * pl.cl; out16[12] = int64_t(pl.main.band_size) * pl.cl;
  out16[13] = int64_t(pl.total_bytes); out16[14] = pl.main.rounds; out16[15] = pl.n_clusters;
  return LR_OK;
}

extern "C" int lr_flatip_plan_passes_sharded(int64_t Q, int64_t N, int k, int64_t d_used, int n_shards, int64_t* out_rows,
                                             int max_passes, int64_t* out_flags2) {
  LR_CHECK_ARG(out_rows && out_flags2 && max_passes >= 1 && Q >= 1 && N >= 1 && k >= 1 && k <= 2048 && d_used >= 1 &&
                   n_shards >= 1, "flatip_plan_passes: bad arguments");
  const FlatipPlan pl = make_plan(Q, N, k, d_used, n_shards);
  int n = 0;
  auto put = [&](const PassPlan& pp) {
    if (n < max_passes) {
      out_rows[4 * n + 0] = pp.tile_begin; out_rows[4 * n + 1] = pp.tile_end;
      out_rows[4 * n + 2] = pp.splits; out_rows[4 * n + 3] = pp.sched;
    }
    ++n;
  };
  if (pl.prefix.units > 0) put(pl.prefix);
  for (int i = 0; i < pl.n_mid; ++i) put(pl.mid[i]);
  put(pl.main);
  out_flags2[0] = pl.wide; out_flags2[1] = pl.lmul;
  return n;
}

extern "C" int lr_flatip_plan_passes(int64_t Q, int64_t N, int k, int64_t d_used, int64_t* out_rows, int max_passes,
                                     int64_t* out_flags2) {
  return lr_flatip_plan_passes_sharded(Q, N, k, d_used, 1, out_rows, max_passes, out_flags2);
}

extern "C" int lr_flatip_last_plan_passes(int64_t* out_rows, int max_passes) {
  LR_CHECK_ARG(out_rows && max_passes >= 1, "flatip_last_plan_passes: bad arguments");
  const FlatipPlan& pl = g_last_plan;
  int n = 0;
  auto put = [&](const PassPlan& pp) {
    if (n < max_passes) {
      out_rows[4 * n + 0] = pp.tile_begin; out_rows[4 * n + 1] = pp.tile_end;
      out_rows[4 * n + 2] = pp.splits; out_rows[4 * n + 3] = pp.sched;
    }
    ++n;
  };
  if (pl.prefix.units > 0) put(pl.prefix);
  for (int i = 0; i < pl.n_mid; ++i) put(pl.mid[i]);
  if (pl.main.units > 0) put(pl.main);
  return n;
}

extern "C" int lr_flatip_last_plan(int64_t* out8) {
  const FlatipPlan& pl = g_last_plan;
  out8[0] = pl.m_tiles; out8[1] = pl.n_tiles; out8[2] = pl.main.splits; out8[3] = pl.main.band_size * pl.cl;
  out8[4] = pl.cap; out8[5] = pl.main.grid * pl.cl; out8[6] = pl.main.units; out8[7] = pl.prefix.tile_end;
  return LR_OK;
}

// One search = phase A (warm-start prefix -> `carry` + thresholds) then the refresh passes and the main pass.  The
// unsharded entry point runs both; a row-sharded search runs them as two calls with the caller's exchange of the
// per-shard prefix top-k in between (RUN_PREFIX writes prefix_keys_out, RUN_REST reads seed_keys).
enum { RUN_PREFIX = 1, RUN_REST = 2 };
// Filters (live / allow / q_filter, all null for the unfiltered entry points) reach every pass: the prefix, the refresh
// passes and the main pass list allowed documents only, so the carried top-k, the thresholds it seeds and the prefix keys
// a sharded search exchanges are all taken over the allowed set.
static int flatip_run(int phases, int shards, const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q,
                      int64_t N, int64_t d_used, const float* q_scale, const float* c_scale, int64_t id_offset, int k,
                      uint64_t* prefix_keys_out, const uint64_t* seed_keys, float* out_scores, int64_t* out_ids,
                      uint64_t* out_keys, const uint32_t* live, const uint32_t* allow, int64_t ld_words, int n_filters,
                      const int32_t* q_filter, void* workspace, size_t ws_bytes, void* stream) {
  int rc = check_flatip_args(q, ldq, corpus, ldc, Q, N, d_used);
  if (rc) return rc;
  LR_CHECK_ARG(k >= 1 && k <= 2048, "flatip: k (%d) must be in [1, 2048]", k);
  LR_CHECK_ARG(shards >= 1 && shards <= 1024, "flatip: n_shards (%d) must be in [1, 1024]", shards);
  LR_CHECK_ARG(id_offset >= 0 && id_offset + N <= (int64_t(1) << 32) - 2, "flatip: id_offset + N must stay below 2^32");
  DocFilter flt;
  if ((rc = make_doc_filter(live, allow, ld_words, n_filters, q_filter, id_offset, N, flt))) return rc;
  if (phases & RUN_REST) LR_CHECK_ARG(out_scores || out_ids || out_keys, "flatip: no output requested");
  const FlatipPlan& pl = make_plan(Q, N, k, d_used, shards);
  if (!workspace || ws_bytes < pl.total_bytes || (uintptr_t(workspace) & 255)) {
    set_error("flatip: workspace too small or misaligned (%zu given, %zu needed, 256-byte aligned)", ws_bytes,
              pl.total_bytes);
    return LR_EWORKSPACE;
  }
  g_last_plan = pl;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUtensorMap tmA, tmB;
  if ((rc = make_tmap(&tmA, q, Q, d_used, ldq, BM))) return rc;
  if ((rc = make_tmap(&tmB, corpus, N, d_used, ldc, BN / pl.cl))) return rc;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  uint32_t* gthr = reinterpret_cast<uint32_t*>(ws + pl.off_gthr);
  int32_t* counts = reinterpret_cast<int32_t*>(ws + pl.off_counts);
  uint64_t* cand = reinterpret_cast<uint64_t*>(ws + pl.off_cand);
  const bool two_phase = pl.prefix.units > 0;

  GemmParams prm{};
  prm.k = k; prm.cap = pl.cap;
  prm.q_scale = q_scale; prm.c_scale = c_scale;
  prm.gthr = gthr;
  prm.filter = flt;
  const ProfileEvents pe_saved = profile_events();
  uint64_t* carry = reinterpret_cast<uint64_t*>(ws + pl.off_carry);  // merged top-k so far: [q_pad][cap], k used
  bool first_rest_pass = true;
  auto run_pass = [&](const PassPlan& pp, bool last) -> int {
    // carried top-k -> list slot `pp.splits` of the candidate array (+ thresholds), the pass, then the merge
    const int own_lists = pp.splits * pl.lmul;
    uint64_t* slot = cand + size_t(own_lists) * pl.q_pad * pl.cap;
    if (two_phase) {
      // the exchanged k-th best of the whole prefix seeds the first pass after the exchange
      const uint64_t* seed = first_rest_pass ? seed_keys : nullptr;
      carry_topk_kernel<<<unsigned(pl.q_pad), 128, 0, st>>>(carry, pl.cap, k, pl.q_pad, Q, slot, gthr,
                                                            counts + size_t(own_lists) * pl.q_pad, seed);
      LR_LAUNCH_CHECK();
    }
    first_rest_pass = false;
    fill_params(prm, pl, pp, Q, N, d_used);
    if (pp.sched) {
      prm.team_ctr = reinterpret_cast<uint32_t*>(ws + pl.off_teamctr);
      LR_CUDA(cudaMemsetAsync(prm.team_ctr, 0, size_t(pp.n_bands) * size_t(pl.n_clusters) * 4, st));
    }
    prm.counts = counts;
    prm.cand = cand;
    if (!last) profile_events() = ProfileEvents{};  // the profiling events bracket the main pass only
    int r = launch_pass<EPI_TOPK>(pl, pp, tmA, tmB, prm, st);
    profile_events() = pe_saved;
    if (r) return r;
    const int lists = own_lists + (two_phase ? 1 : 0);
    if (last)
      return topk_merge_two_level(cand, counts, lists, Q, pl.q_pad, pl.cap, k, LR_SCORE_F32, id_offset, out_scores, out_ids,
                                  out_keys, k, ws + pl.off_merge, pl.merge_bytes, st);
    return topk_merge_two_level(cand, counts, lists, Q, pl.q_pad, pl.cap, k, LR_SCORE_F32, 0, nullptr, nullptr, carry,
                                pl.cap, ws + pl.off_merge, pl.merge_bytes, st);
  };
  if (phases & RUN_PREFIX) {
    if (two_phase) {
      // ---- phase A: prefix -> merged top-k in `carry`
      profile_events() = ProfileEvents{};
      fill_params(prm, pl, pl.prefix, Q, N, d_used);
      prm.counts = reinterpret_cast<int32_t*>(ws + pl.off_pcounts);
      prm.cand = reinterpret_cast<uint64_t*>(ws + pl.off_pcand);
      LR_CUDA(cudaMemsetAsync(gthr, 0, size_t(pl.q_pad) * 4, st));
      rc = launch_pass<EPI_TOPK>(pl, pl.prefix, tmA, tmB, prm, st);
      if (!rc)
        rc = topk_merge_two_level(prm.cand, prm.counts, pl.prefix.splits * pl.lmul, Q, pl.q_pad, pl.cap, k, LR_SCORE_F32, 0,
                                  nullptr, nullptr, carry, pl.cap, ws + pl.off_merge, pl.merge_bytes, st);
      profile_events() = pe_saved;
      if (rc) return rc;
      if (prefix_keys_out)
        LR_CUDA(cudaMemcpy2DAsync(prefix_keys_out, size_t(k) * 8, carry, size_t(pl.cap) * 8, size_t(k) * 8, size_t(Q),
                                  cudaMemcpyDeviceToDevice, st));
    } else {
      LR_CUDA(cudaMemsetAsync(gthr, 0, size_t(pl.q_pad) * 4, st));
      if (prefix_keys_out) LR_CUDA(cudaMemsetAsync(prefix_keys_out, 0, size_t(Q) * size_t(k) * 8, st));
    }
  }
  if (!(phases & RUN_REST)) return LR_OK;
  if (!two_phase && seed_keys) {  // single-phase plan of a sharded search: the seed is the only warm start
    seed_thresholds_kernel<<<unsigned((Q + 255) / 256), 256, 0, st>>>(seed_keys, k, Q, gthr);
    LR_LAUNCH_CHECK();
  }
  // ---- threshold-refresh passes (epilogue-bound searches only), then phase B / single phase
  for (int i = 0; i < pl.n_mid; ++i)
    if ((rc = run_pass(pl.mid[i], false))) return rc;
  return run_pass(pl.main, true);
}

extern "C" int lr_flatip_topk(const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q, int64_t N,
                              int64_t d_used, const float* q_scale, const float* c_scale, int64_t id_offset, int k,
                              float* out_scores, int64_t* out_ids, uint64_t* out_keys, void* workspace,
                              size_t ws_bytes, void* stream) {
  return flatip_run(RUN_PREFIX | RUN_REST, 1, q, ldq, corpus, ldc, Q, N, d_used, q_scale, c_scale, id_offset, k, nullptr,
                    nullptr, out_scores, out_ids, out_keys, nullptr, nullptr, 0, 0, nullptr, workspace, ws_bytes, stream);
}

extern "C" int lr_flatip_topk_filtered(const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q, int64_t N,
                                       int64_t d_used, const float* q_scale, const float* c_scale, int64_t id_offset,
                                       int k, float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                                       const uint32_t* live, const uint32_t* allow, int64_t ld_words, int n_filters,
                                       const int32_t* q_filter, void* workspace, size_t ws_bytes, void* stream) {
  return flatip_run(RUN_PREFIX | RUN_REST, 1, q, ldq, corpus, ldc, Q, N, d_used, q_scale, c_scale, id_offset, k, nullptr,
                    nullptr, out_scores, out_ids, out_keys, live, allow, ld_words, n_filters, q_filter, workspace,
                    ws_bytes, stream);
}

extern "C" size_t lr_flatip_workspace_bytes_sharded(int64_t Q, int64_t N, int k, int64_t d_used, int n_shards) {
  if (Q < 1 || N < 1 || k < 1 || d_used < 1 || n_shards < 1) return 0;
  return make_plan(Q, N, k, d_used, n_shards).total_bytes;
}

extern "C" int lr_flatip_topk_begin(const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q, int64_t N,
                                    int64_t d_used, const float* q_scale, const float* c_scale, int k, int n_shards,
                                    uint64_t* out_prefix_keys, void* workspace, size_t ws_bytes, void* stream) {
  LR_CHECK_ARG(out_prefix_keys, "flatip_topk_begin: null out_prefix_keys");
  return flatip_run(RUN_PREFIX, n_shards, q, ldq, corpus, ldc, Q, N, d_used, q_scale, c_scale, 0, k, out_prefix_keys,
                    nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, nullptr, workspace, ws_bytes, stream);
}

extern "C" int lr_flatip_topk_begin_filtered(const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q,
                                             int64_t N, int64_t d_used, const float* q_scale, const float* c_scale,
                                             int64_t id_offset, int k, int n_shards, uint64_t* out_prefix_keys,
                                             const uint32_t* live, const uint32_t* allow, int64_t ld_words,
                                             int n_filters, const int32_t* q_filter, void* workspace, size_t ws_bytes,
                                             void* stream) {
  LR_CHECK_ARG(out_prefix_keys, "flatip_topk_begin: null out_prefix_keys");
  return flatip_run(RUN_PREFIX, n_shards, q, ldq, corpus, ldc, Q, N, d_used, q_scale, c_scale, id_offset, k,
                    out_prefix_keys, nullptr, nullptr, nullptr, nullptr, live, allow, ld_words, n_filters, q_filter,
                    workspace, ws_bytes, stream);
}

extern "C" int lr_flatip_topk_finish(const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q, int64_t N,
                                     int64_t d_used, const float* q_scale, const float* c_scale, int64_t id_offset,
                                     int k, int n_shards, const uint64_t* seed_keys, float* out_scores,
                                     int64_t* out_ids, uint64_t* out_keys, void* workspace, size_t ws_bytes,
                                     void* stream) {
  return flatip_run(RUN_REST, n_shards, q, ldq, corpus, ldc, Q, N, d_used, q_scale, c_scale, id_offset, k, nullptr,
                    seed_keys, out_scores, out_ids, out_keys, nullptr, nullptr, 0, 0, nullptr, workspace, ws_bytes,
                    stream);
}

extern "C" int lr_flatip_topk_finish_filtered(const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q,
                                              int64_t N, int64_t d_used, const float* q_scale, const float* c_scale,
                                              int64_t id_offset, int k, int n_shards, const uint64_t* seed_keys,
                                              float* out_scores, int64_t* out_ids, uint64_t* out_keys,
                                              const uint32_t* live, const uint32_t* allow, int64_t ld_words,
                                              int n_filters, const int32_t* q_filter, void* workspace, size_t ws_bytes,
                                              void* stream) {
  return flatip_run(RUN_REST, n_shards, q, ldq, corpus, ldc, Q, N, d_used, q_scale, c_scale, id_offset, k, nullptr,
                    seed_keys, out_scores, out_ids, out_keys, live, allow, ld_words, n_filters, q_filter, workspace,
                    ws_bytes, stream);
}

extern "C" int lr_flatip_scores(const void* q, int64_t ldq, const void* corpus, int64_t ldc, int64_t Q, int64_t N,
                                int64_t d_used, float* out_scores, void* stream) {
  int rc = check_flatip_args(q, ldq, corpus, ldc, Q, N, d_used);
  if (rc) return rc;
  LR_CHECK_ARG(out_scores, "flatip_scores: null output");
  FlatipPlan pl = make_plan(Q, N, 1, 4096);
  const PassPlan all = plan_pass(pl.m_groups, pl.n_clusters, 0, pl.n_tiles, 1 << 20, 0);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUtensorMap tmA, tmB;
  if ((rc = make_tmap(&tmA, q, Q, d_used, ldq, BM))) return rc;
  if ((rc = make_tmap(&tmB, corpus, N, d_used, ldc, BN / pl.cl))) return rc;
  GemmParams prm{};
  fill_params(prm, pl, all, Q, N, d_used);
  prm.dbg_scores = out_scores;
  return launch_pass<EPI_STORE>(pl, all, tmA, tmB, prm, st);
}
