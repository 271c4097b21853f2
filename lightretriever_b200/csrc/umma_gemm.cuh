// umma_gemm.cuh — the TMA -> tcgen05.mma -> TMEM main loop shared by K2 (flat inner-product top-k) and
// K3 (document sparse head), with the epilogue that makes each of them a fused kernel.
//
// One persistent CTA per SM, warp-specialised:
//   warp 0      TMA producer   (cp.async.bulk.tensor, 128B-swizzled K-major tiles, 4-stage ring)
//   warp 1      MMA issuer     (one thread, tcgen05.mma cta_group::1 kind::f16, M=128 N=256 K=16)
//   warps 2..5  epilogue       (tcgen05.ld 32x32b: one accumulator row per thread)
//   warps 6..9  second epilogue set (WIDE variant only: short rows, where a tile's epilogue outlasts its MMAs; the two
//               sets take alternate tiles = alternate accumulator buffers and keep separate candidate lists)
// The 128x256 f32 accumulator lives in TMEM, double buffered (2 x 256 columns), so the epilogue of
// tile i overlaps the MMAs of tile i+1.  D = A . B^T with A = [rows, K] and B = [cols, K], both K-major bf16.
//
// Work decomposition: unit = (row tile of 128 rows, column split).  Units are ordered
// (band of row tiles, split, row tile in band) and dealt round-robin to the CTAs, so the CTAs running
// concurrently share `band` row tiles (L2-resident) and stream the same few column splits in lock step
// (each B tile is fetched from HBM once per band and hit in L2 by the other CTAs of the band).
//
// Epilogues
//   EPI_STORE   plain f32 store of the tile (debug / parity of the main loop)
//   EPI_TOPK    K2: rows = queries, columns = documents.  Every thread compares its row's scores with a
//               running threshold and appends the survivors to a per-(split,query) candidate list; a full
//               list is cut back to its exact top-k by a warp-cooperative radix select.  The score matrix
//               never reaches HBM.
//   EPI_MAXTOK  K3: rows = vocabulary entries, columns = document tokens.  Every thread keeps the running
//               masked max over the tokens of the current document and writes relu/log1p of it when the
//               document ends (max_linear_map.py:72-85 + modeling_hybrid.py:183-187 in one pass).
#pragma once
#include "common.cuh"

#include <cudaTypedefs.h>
#include <math.h>
#include <mutex>

namespace lr {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;  // 64 bf16 = 128 bytes = one swizzle row
constexpr int A_BYTES = BM * BK * 2;
constexpr int B_BYTES = BN * BK * 2;
constexpr int PIPE_BYTES = 4 * (A_BYTES + B_BYTES);  // shared memory of the operand ring (192 KB)
// cta_group::1 (single CTA or multicast cluster): a stage holds A (16 KB) + the whole B tile (32 KB): 4 stages.
// cta_group::2 (CTA pair, one M=256 MMA): a stage holds A (16 KB) + this CTA's HALF of B (16 KB): 6 stages.
// BIGLIST (top-k with long candidate lists, k > 352): one 48 KB stage (two 32 KB stages for a pair) is given to the
// epilogue warps' list-staging area instead, so that lists of up to 2304 (2816) entries are still cut in shared memory.
// WIDE (top-k with short rows, d_used <= 768, where a tile's epilogue outlasts its MMAs): EIGHT epilogue warps in two
// sets that take alternate tiles (set = accumulator buffer), each with its own candidate lists; one ring stage is given
// to the second set's histograms, column scales and list staging.
template <bool PAIR, bool BIGLIST, bool WIDE = false> struct PipeCfg {
  static_assert(!(BIGLIST && WIDE), "WIDE is for short lists");
  static constexpr int kBBytes = PAIR ? B_BYTES / 2 : B_BYTES;
  static constexpr int kStageBytes = A_BYTES + kBBytes;
  static constexpr int kStages = PIPE_BYTES / kStageBytes - (BIGLIST ? (PAIR ? 2 : 1) : 0) - (WIDE ? 1 : 0);
  static constexpr int kPipeBytes = kStages * kStageBytes;
};
constexpr int GEMM_THREADS = 192;
constexpr int GEMM_THREADS_WIDE = 320;
constexpr int TMEM_COLS = 512;
constexpr int ACC_STAGES = 2;
constexpr int SMEM_BAR_BYTES = 256;
constexpr int SMEM_HIST_BYTES = 4 * 256 * 4;
constexpr int LIST_STAGE_ENTRIES = 768;  // per epilogue warp: a candidate list of <= 768 entries is compacted in smem
constexpr int SMEM_LIST_BYTES = 4 * LIST_STAGE_ENTRIES * 8;
template <bool PAIR, bool BIGLIST, bool WIDE = false> struct ListCfg {
  static constexpr int kWarps = WIDE ? 8 : 4;  // epilogue warps
  // what the ring left, minus the second set's histograms and column scales
  static constexpr int kListBytes = SMEM_LIST_BYTES + (PIPE_BYTES - PipeCfg<PAIR, BIGLIST, WIDE>::kPipeBytes) -
                                    (WIDE ? SMEM_HIST_BYTES + 4 * 256 * 4 : 0);
  static constexpr int kEntries = kListBytes / (kWarps * 8);
};
constexpr int SMEM_CS_BYTES = 4 * BN * 4;  // per epilogue warp: the column scales of the current tile
constexpr int GEMM_SMEM_TOTAL =
    1024 + PIPE_BYTES + SMEM_BAR_BYTES + SMEM_HIST_BYTES + SMEM_LIST_BYTES + SMEM_CS_BYTES;
static_assert(GEMM_SMEM_TOTAL <= 227 * 1024, "shared memory budget exceeded");

enum { EPI_STORE = 0, EPI_TOPK = 1, EPI_MAXTOK = 2 };

struct GemmParams {
  int64_t rows, cols, row_pad;  // rows of A (queries / vocab), rows of B (documents / tokens)
  int kblocks;
  int m_tiles, splits, band_size, n_bands, units;  // band_size / n_bands / units count GROUPS of CL row tiles
  int m_groups;                                    // ceil(m_tiles / CL): one group per cluster
  // Team schedule (sched == 1): inside a band the clusters form fixed teams of (groups in the band) clusters; a team
  // walks its splits together, every member owning one row group, and a progress counter per (band, split) keeps the
  // members within `team_window` tiles of each other so that a B tile is fetched from HBM once per team.
  int sched;
  int team_window;
  uint32_t* team_ctr;  // [n_bands * n_clusters] tiles issued per (band, team), zeroed before the launch
  // column split geometry: split s covers columns [s*cols_per_split_num/den ...) — see split_cols()
  int n_tiles;          // EPI_STORE / EPI_TOPK: 256-column tiles, split = balanced tile range of [tile_begin, n_tiles)
  int tile_begin;
  int64_t seg_len;      // EPI_MAXTOK: tokens per document (S); split = segs_per_split documents
  int64_t n_segs;
  int segs_per_split;
  // EPI_MAXTOK, packed tokens (cu_seqlens != null): document b = columns [cu_seqlens[b], cu_seqlens[b+1]).  Splits are
  // balanced ranges of whole 256-token tiles (n_tiles / tile_begin as for the top-k epilogue), so a document can start in
  // one split and end in another: split_doc0[s] = the document holding the first token of split s (0 for s = 0), and a
  // unit leaves the running max of such a document's piece in edge[(2 s + which) * rows + row] — which = 0 for a
  // document that began before the split, 1 for one that goes on after it — for sparse_head_fix_kernel to combine.
  const int32_t* cu_seqlens;
  const int32_t* split_doc0;
  float* edge;
  // EPI_TOPK
  int k, cap;
  const float* q_scale;
  const float* c_scale;
  uint64_t* cand;    // [splits][row_pad][cap]
  int32_t* counts;   // [splits][row_pad]
  uint32_t* gthr;    // [row_pad] shared lower bound on each query's k-th best score (key space)
  DocFilter filter;  // documents a query may return (filter.on == 0: all); applied before a score enters a list
  // EPI_STORE
  float* dbg_scores; // [rows][cols]
  // EPI_MAXTOK
  const float* bias;      // [rows] or null
  const uint8_t* mask;    // [cols] 1 = valid token
  float* out;             // [n_segs][rows]
  int relu, log1p;
};

// unit u -> (group of CL row tiles, column split)
__device__ __forceinline__ void decode_unit(const GemmParams& p, int u, int& m_group, int& split) {
  const int per_band = p.band_size * p.splits;
  int b = u / per_band;
  if (b > p.n_bands - 1) b = p.n_bands - 1;
  const int rem = u - b * per_band;
  const int mb = min(p.band_size, p.m_groups - b * p.band_size);
  split = rem / mb;
  m_group = b * p.band_size + rem % mb;
}
// Visit the units of one cluster: f(m_group, split, team_size, ctr_index).  All three warp roles walk the same sequence.
template <class F>
__device__ __forceinline__ void for_each_unit(const GemmParams& p, int cluster_id, int n_clusters, F&& f) {
  if (p.sched == 0) {  // round robin over (band, split, group in band)
    for (int u = cluster_id; u < p.units; u += n_clusters) {
      int m_group, split;
      decode_unit(p, u, m_group, split);
      f(m_group, split, 1, 0);
    }
  } else {  // fixed teams per band
    for (int b = 0; b < p.n_bands; ++b) {
      const int mb = min(p.band_size, p.m_groups - b * p.band_size);
      const int n_teams = n_clusters / mb;
      const int team = cluster_id / mb, g = cluster_id - team * mb;
      if (team >= n_teams) continue;  // this cluster sits the band out
      for (int split = team; split < p.splits; split += n_teams) f(b * p.band_size + g, split, mb, b * n_clusters + team);
    }
  }
}

// columns [c0, c1) covered by a split; tiles start at c0 and step BN
template <int EPI>
__device__ __forceinline__ void split_cols(const GemmParams& p, int split, int64_t& c0, int64_t& c1) {
  if (EPI == EPI_MAXTOK && p.cu_seqlens == nullptr) {
    const int64_t s0 = int64_t(split) * p.segs_per_split;
    int64_t s1 = s0 + p.segs_per_split;
    if (s1 > p.n_segs) s1 = p.n_segs;
    c0 = s0 * p.seg_len;
    c1 = s1 * p.seg_len;
  } else {
    const int64_t nt = p.n_tiles - p.tile_begin;
    const int64_t t0 = p.tile_begin + (int64_t(split) * nt) / p.splits;
    const int64_t t1 = p.tile_begin + (int64_t(split + 1) * nt) / p.splits;
    c0 = t0 * BN;
    c1 = t1 * BN;
    if (c1 > p.cols) c1 = p.cols;
  }
}

// Cut a candidate list (n entries, ascending id order) back to its exact top-k, keeping id order.
// Returns the score key of the k-th best entry.  All 32 lanes participate.
// When the list fits the warp's shared-memory staging area it is pulled in with one coalesced sweep, the four radix
// passes and the stable compaction run on shared memory, and only the survivors go back to global memory; otherwise
// every pass re-reads the list from L2.
static __device__ __noinline__ uint32_t warp_compact_topk(uint64_t* buf, int n, int k, uint32_t* hist,
                                                          uint64_t* stage, int stage_cap, int lane) {
  const uint32_t full = 0xFFFFFFFFu;
  const bool staged = n <= stage_cap;
  if (staged) {
    for (int i = lane; i < n; i += 32) stage[i] = ld_cg_u64(buf + i);
    __syncwarp();
  }
  uint32_t prefix = 0;
  uint32_t remaining = uint32_t(k);
#pragma unroll 1
  for (int pass = 3; pass >= 0; --pass) {
    const int shift = pass * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) hist[lane * 8 + i] = 0;
    __syncwarp();
    for (int i = lane; i < n; i += 32) {
      const uint32_t h = key_hi(staged ? stage[i] : ld_cg_u64(buf + i));
      const bool match = (pass == 3) || ((h >> (shift + 8)) == prefix);
      if (match) atomicAdd(&hist[(h >> shift) & 0xFFu], 1u);
    }
    __syncwarp();
    uint32_t bin, rem2;
    bool take_all;
    warp_find_bin_desc(hist, remaining, bin, rem2, take_all);
    prefix = (prefix << 8) | bin;
    remaining = rem2;
    __syncwarp();
  }
  const uint32_t vk = prefix;            // score key of the k-th best
  const uint32_t keep_ties = remaining;  // how many entries equal to vk survive (lowest ids first)
  // stable compaction (in place: the write index never passes the read index)
  uint32_t out = 0, ties_seen = 0;
  const uint32_t lt = lanemask_lt();
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    const bool in = i < n;
    const uint64_t key = in ? (staged ? stage[i] : ld_cg_u64(buf + i)) : 0ull;
    const uint32_t h = key_hi(key);
    const bool gt = in && h > vk;
    const bool eq = in && h == vk;
    const uint32_t eqm = __ballot_sync(full, eq);
    const uint32_t tie_rank = ties_seen + __popc(eqm & lt);
    const bool keep = gt || (eq && tie_rank < keep_ties);
    const uint32_t km = __ballot_sync(full, keep);
    if (keep) st_cg_u64(buf + out + __popc(km & lt), key);
    out += __popc(km);
    ties_seen += __popc(eqm);
  }
  __syncwarp();
  return vk;
}

// v[j] for a per-thread dynamic j in [0, 32): 16+8+4+2+1 selects, no branches, no local memory
__device__ __forceinline__ uint32_t select32(const uint32_t (&v)[32], int j) {
  uint32_t a[16], b[8], c[4], d[2];
  const bool b0 = j & 1, b1 = j & 2, b2 = j & 4, b3 = j & 8, b4 = j & 16;
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = b0 ? v[2 * i + 1] : v[2 * i];
#pragma unroll
  for (int i = 0; i < 8; ++i) b[i] = b1 ? a[2 * i + 1] : a[2 * i];
#pragma unroll
  for (int i = 0; i < 4; ++i) c[i] = b2 ? b[2 * i + 1] : b[2 * i];
#pragma unroll
  for (int i = 0; i < 2; ++i) d[i] = b3 ? c[2 * i + 1] : c[2 * i];
  return b4 ? d[1] : d[0];
}

constexpr float BF16_LOWEST = -3.3895313892515355e38f;  // torch.finfo(torch.bfloat16).min
// Longest a producer waits for its team (about 2-3 ms; a full-width tile takes ~30k cycles, so a live team is never this
// far apart).  After one timeout the cluster stops pacing itself for the rest of the launch.
constexpr long long TEAM_WAIT_CYCLES = 4ll * 1000 * 1000;

// CL = CTAs per cluster (1 or 2).  With CL == 2 the two CTAs own adjacent row tiles of the same column split; each
// loads its own A tile and HALF of the shared B tile, multicast into both CTAs' shared memory, so the L2 -> SM
// traffic per CTA and k-block drops from 48 KB to 32 KB.  tmB's box then holds BN / CL rows.
// PAIR (requires CL == 2): the two CTAs form one cta_group::2 MMA — M = 256 (128 rows per CTA), each CTA stores its A
// tile and HALF of B (the tensor cores read both halves), the leader CTA's thread issues the MMAs for both, TMA
// completions of both CTAs are counted on the leader's full barrier, commits are multicast to both CTAs.
template <int EPI, int CL, bool PAIR, bool BIGLIST, bool WIDE>
__global__ void __launch_bounds__(WIDE ? GEMM_THREADS_WIDE : GEMM_THREADS, 1)
umma_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const GemmParams p) {
  static_assert(!PAIR || CL == 2, "cta_group::2 needs a cluster of two CTAs");
  static_assert(!WIDE || EPI == EPI_TOPK, "the two-set epilogue exists for the top-k epilogue only");
  constexpr int STAGES = PipeCfg<PAIR, BIGLIST, WIDE>::kStages;
  constexpr int STAGE_BYTES = PipeCfg<PAIR, BIGLIST, WIDE>::kStageBytes;
  constexpr int kPipe = PipeCfg<PAIR, BIGLIST, WIDE>::kPipeBytes;
  constexpr int kListEntries = ListCfg<PAIR, BIGLIST, WIDE>::kEntries;
  constexpr int NEPI = ListCfg<PAIR, BIGLIST, WIDE>::kWarps;
  // shared memory map: operand ring | barriers | histograms | column scales | list staging (takes what the ring left)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + kPipe;
  // barrier map (8 bytes each): full[STAGES], empty[STAGES], tfull[2], tempty[2], then the TMEM pointer slot
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + ACC_STAGES + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 2 * ACC_STAGES);
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + kPipe + 8 * (2 * STAGES + 2 * ACC_STAGES));
  uint32_t* hist_all = reinterpret_cast<uint32_t*>(smem_gen + kPipe + SMEM_BAR_BYTES);
  float* cs_all = reinterpret_cast<float*>(smem_gen + kPipe + SMEM_BAR_BYTES + NEPI * 256 * 4);
  uint64_t* list_stage_all =
      reinterpret_cast<uint64_t*>(smem_gen + kPipe + SMEM_BAR_BYTES + NEPI * 256 * 4 + NEPI * BN * 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta_rank = (CL > 1) ? int(cluster_ctarank()) : 0;
  const int cluster_id = int(blockIdx.x) / CL;
  const int n_clusters = int(gridDim.x) / CL;
  constexpr uint16_t kMcMask = uint16_t((1u << CL) - 1u);

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmA);
    prefetch_tensormap(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      // multicast cluster: every CTA must have consumed the slot; pair: one multicast commit of the leader
      mbar_init(empty_bar(s), PAIR ? 1 : CL);
    }
    for (int s = 0; s < ACC_STAGES; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), PAIR ? 8 : 4);  // one arrive per epilogue warp (of both CTAs for a pair)
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    if (PAIR) {
      tmem_alloc_2sm(tmem_slot, TMEM_COLS);
      tmem_relinquish_2sm();
    } else {
      tmem_alloc(tmem_slot, TMEM_COLS);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();  // peers' barriers are initialised before any multicast can reach them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int team_slot = -1, ti = 0;  // progress counter in use and tiles issued against it (cumulative over the units)
      // The team pacing is a performance hint (L2 reuse of B tiles), never a data dependency: a member that does not show
      // up within TEAM_WAIT_CYCLES (its SM is held by another kernel, MPS, a smaller part) ends the pacing for this
      // cluster — it runs free for the rest of the launch instead of waiting on a CTA that may not be resident.
      bool team_live = true;
      for_each_unit(p, cluster_id, n_clusters, [&](int m_group, int split, int team_size, int ctr_index) {
        int64_t c0, c1;
        const int m_tile = m_group * CL + cta_rank;  // may be a padding tile (>= m_tiles): TMA zero-fills it
        split_cols<EPI>(p, split, c0, c1);
        const bool team_sync = p.sched != 0 && team_size > 1 && cta_rank == 0;
        uint32_t* ctr = team_sync ? p.team_ctr + ctr_index : nullptr;
        if (ctr_index != team_slot) {
          team_slot = ctr_index;
          ti = 0;
        }
        for (int64_t cb = c0; cb < c1; cb += BN, ++ti) {
          if (team_sync && team_live && ti >= p.team_window) {
            // do not run more than team_window tiles ahead of the slowest member of the team
            const uint32_t need = uint32_t(team_size) * uint32_t(ti - p.team_window + 1);
            if (ld_acquire_u32(ctr) < need) {
              const long long t0 = clock64();
              while (ld_acquire_u32(ctr) < need) {
                if (clock64() - t0 > TEAM_WAIT_CYCLES) {
                  team_live = false;
                  break;
                }
              }
            }
          }
          for (int kb = 0; kb < p.kblocks; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            const uint32_t a_dst = smem_base + stage * STAGE_BYTES;
            if (PAIR) {
              // both CTAs' bytes are counted on the leader's barrier; only the leader arms it
              const uint32_t leader_full = mapa_cluster(full_bar(stage), 0);
              if (cta_rank == 0) mbar_arrive_expect_tx(full_bar(stage), 2 * STAGE_BYTES);
              tma_load_2d_2sm(a_dst, &tmA, kb * BK, m_tile * BM, leader_full, L2_EVICT_NORMAL);
              tma_load_2d_2sm(a_dst + A_BYTES, &tmB, kb * BK, int(cb) + cta_rank * (BN / 2), leader_full,
                              L2_EVICT_NORMAL);
              if (++stage == STAGES) {
                stage = 0;
                phase ^= 1u;
              }
              continue;
            }
            mbar_arrive_expect_tx(full_bar(stage), STAGE_BYTES);
            tma_load_2d_hint(a_dst, &tmA, kb * BK, m_tile * BM, full_bar(stage), L2_EVICT_NORMAL);
            if (CL == 1) {
              tma_load_2d_hint(a_dst + A_BYTES, &tmB, kb * BK, int(cb), full_bar(stage), L2_EVICT_NORMAL);
            } else {
              // my half of the B tile, delivered to both CTAs (same offsets, each CTA's own full barrier)
              tma_load_2d_mc_hint(a_dst + A_BYTES + cta_rank * (B_BYTES / CL), &tmB, kb * BK,
                                  int(cb) + cta_rank * (BN / CL), full_bar(stage), kMcMask, L2_EVICT_NORMAL);
            }
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
          if (team_sync) red_release_add_u32(ctr, 1u);  // this member has issued tile ti
        }
      });
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (single thread)
    if (lane == 0 && (!PAIR || cta_rank == 0)) {  // pair: the leader CTA issues for both
      constexpr uint32_t idesc = umma_idesc_bf16(PAIR ? 2 * BM : BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for_each_unit(p, cluster_id, n_clusters, [&](int m_group, int split, int, int) {
        (void)m_group;
        int64_t c0, c1;
        split_cols<EPI>(p, split, c0, c1);
        for (int64_t cb = c0; cb < c1; cb += BN) {
          mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + uint32_t(acc * BN);
          for (int kb = 0; kb < p.kblocks; ++kb) {
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            const uint32_t a_addr = smem_base + stage * STAGE_BYTES;
            const uint64_t a_desc = umma_desc_k_sw128(a_addr);
            const uint64_t b_desc = umma_desc_k_sw128(a_addr + A_BYTES);
#pragma unroll
            for (int kk = 0; kk < BK / 16; ++kk) {
              // +32 bytes per K=16 step inside the 128-byte swizzle row: +2 in the (addr >> 4) field
              if (PAIR)
                umma_bf16_2sm(d_tmem, a_desc + uint64_t(kk * 2), b_desc + uint64_t(kk * 2), idesc,
                              (kb | kk) != 0 ? 1u : 0u);
              else
                umma_bf16(d_tmem, a_desc + uint64_t(kk * 2), b_desc + uint64_t(kk * 2), idesc,
                          (kb | kk) != 0 ? 1u : 0u);
            }
            // the smem slot is free once these MMAs have read it — in every CTA the multicast writes to
            if (PAIR) umma_commit_2sm_mc(empty_bar(stage), kMcMask);
            else if (CL == 1) umma_commit(empty_bar(stage));
            else umma_commit_mc(empty_bar(stage), kMcMask);
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
          // accumulator complete -> epilogue (of both CTAs for a pair)
          if (PAIR) umma_commit_2sm_mc(tfull_bar(acc), kMcMask);
          else umma_commit(tfull_bar(acc));
          if (++acc == ACC_STAGES) {
            acc = 0;
            acc_phase ^= 1u;
          }
        }
      });
    }
  } else {
    // ------------------------------------------------------------ epilogue warps (TMEM lane quarter = warp % 4)
    const int quarter = warp & 3;
    const int row_in_tile = quarter * 32 + lane;
    const int eset = WIDE ? (warp - 2) >> 2 : 0;  // WIDE: set 0 drains accumulator buffer 0 (even tiles), set 1 buffer 1
    uint32_t* hist = hist_all + (warp - 2) * 256;
    uint64_t* list_stage = list_stage_all + (warp - 2) * kListEntries;
    float* cs_smem = cs_all + (warp - 2) * BN;
    int64_t tiles_before = 0;  // tiles of the earlier units of this cluster: the accumulator buffers alternate globally
    const bool has_scale = (EPI == EPI_TOPK) && (p.q_scale != nullptr || p.c_scale != nullptr);
    const uint32_t full = 0xFFFFFFFFu;
    int acc = WIDE ? eset : 0;
    uint32_t acc_phase = 0;
    for_each_unit(p, cluster_id, n_clusters, [&](int m_group, int split, int, int) {
      int64_t c0, c1;
      const int m_tile = m_group * CL + cta_rank;
      split_cols<EPI>(p, split, c0, c1);
      const int list_idx = WIDE ? split * 2 + eset : split;  // candidate list of this (unit, epilogue set)
      constexpr int64_t TILE_STEP = WIDE ? 2 * BN : BN;
      // first tile of the unit that this set owns
      const int64_t cfirst = c0 + ((WIDE && int(tiles_before & 1) != eset) ? BN : 0);
      tiles_before += (c1 - c0 + BN - 1) / BN;
      const int64_t row = int64_t(m_tile) * BM + row_in_tile;
      const bool row_valid = row < p.rows;
      const bool tile_valid = m_tile < p.m_tiles;  // false only for the padding tile of an odd last group
      // EPI_TOPK per-row running state
      uint64_t* buf = nullptr;
      uint32_t cnt = 0;
      float thr_local = -INFINITY;
      float qs = 1.0f;
      // EPI_MAXTOK per-row running state
      float run_max = BF16_LOWEST;
      float bias_v = 0.0f;
      int64_t seg = 0, seg_end = 0, seg_stop = 0, next_end = 0;
      bool head_open = false;  // packed: the first document of the unit began in an earlier split (its piece goes to `edge`)
      float head_piece = BF16_LOWEST;
      if (EPI == EPI_TOPK && tile_valid) {
        buf = p.cand + (int64_t(list_idx) * p.row_pad + row) * p.cap;
        if (row_valid && p.q_scale) qs = p.q_scale[row];
      }
      if (EPI == EPI_MAXTOK) {
        if (row_valid && p.bias) bias_v = p.bias[row];
        if (p.cu_seqlens) {  // the end after next is fetched one document ahead of its use
          seg = p.split_doc0[split];
          head_open = int64_t(p.cu_seqlens[seg]) < c0;
          seg_end = p.cu_seqlens[seg + 1];
          next_end = p.cu_seqlens[min(seg + 2, p.n_segs)];
        } else {
          seg = int64_t(split) * p.segs_per_split;
          seg_stop = min(seg + p.segs_per_split, p.n_segs);
          seg_end = c0 + p.seg_len;
        }
      }
      // a document is complete: its activation goes to `out` — or, for the piece of a document that began earlier, the raw
      // max is kept for the edge buffer
      auto emit_doc = [&]() {
        if (head_open) {
          head_piece = run_max;
          head_open = false;
        } else {
          float x = run_max;
          if (p.relu) x = fmaxf(x, 0.0f);
          if (p.log1p) x = log1pf(x);
          if (row_valid) p.out[seg * p.rows + row] = x;
        }
        run_max = BF16_LOWEST;
        ++seg;
      };
      // The shared threshold and the column scales of a tile are fetched one tile ahead (a threshold that is one tile
      // stale is still a valid lower bound), so no global latency sits between two tiles of an epilogue-bound pass.
      uint32_t g_pref = 0;
      float cs_pref[BN / 32];
      auto load_cs = [&](int64_t cbx) {
#pragma unroll
        for (int i = 0; i < BN / 32; ++i) {
          const int64_t dcol = cbx + i * 32 + lane;
          cs_pref[i] = (p.c_scale && dcol < p.cols) ? p.c_scale[dcol] : (p.c_scale ? 0.0f : 1.0f);
        }
      };
      if (EPI == EPI_TOPK) {
        if (row_valid) g_pref = ld_relaxed_u32(p.gthr + row);
        if (has_scale && cfirst < c1) load_cs(cfirst);
      }
      for (int64_t cb = cfirst; cb < c1; cb += TILE_STEP) {
        const int n_valid = (c1 - cb < int64_t(BN)) ? int(c1 - cb) : BN;
        float thr = INFINITY;
        if (EPI == EPI_TOPK && row_valid) {
          const uint32_t g = g_pref;
          const float tg = (g <= KEY_NEG_INF) ? -INFINITY : key_to_f32(g - 1u);  // s >= gthr  <=>  s > tg
          thr = fmaxf(thr_local, tg);
        }
        if (EPI == EPI_TOPK && has_scale) {
          // column scales of this tile -> shared memory (read back as broadcasts)
          __syncwarp();
#pragma unroll
          for (int i = 0; i < BN / 32; ++i) cs_smem[i * 32 + lane] = cs_pref[i];
          __syncwarp();
        }
        if (EPI == EPI_TOPK && cb + TILE_STEP < c1) {
          if (row_valid) g_pref = ld_relaxed_u32(p.gthr + row);
          if (has_scale) load_cs(cb + TILE_STEP);
        }
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const uint32_t t_addr = tmem_base + (uint32_t(quarter * 32) << 16) + uint32_t(acc * BN);
        if (EPI == EPI_TOPK) {
          // Software-pipelined over 32-column chunks: while chunk c is compared against the threshold (pure register
          // work), the tcgen05.ld of chunk c+1 is in flight.  A chunk first yields a 32-bit pass mask; the (rare) appends
          // and list cuts run only after the in-flight load has completed.
          const int nchunks = (n_valid + 31) >> 5;
          // Scaled scores (MRL prefixes): the row scale is folded into the threshold, thr_s = thr / qs nudged down, so the
          // filter costs one LDS + FFMA + funnel shift per score (sign of thr_s - v * cs[j]); it may admit a score that
          // is not above the exact threshold, which the append path re-checks with the exact product.
          float thr_s = thr;
          if (has_scale && thr < INFINITY && thr > -INFINITY) {
            thr_s = thr / qs;
            thr_s -= fabsf(thr_s) * 4.8e-7f + 1e-37f;  // 4 ulp: thr_s * qs <= thr in every rounding
          }
          // Pass mask of a chunk from sign bits: d = thr - score is negative exactly when score > thr (thr - s is +0 for
          // s == thr; thr = +inf rejects and thr = -inf admits everything).  One FADD (FFMA with a column scale) and one
          // funnel shift per score, in four independent 8-score chains — the epilogue warp is alone on its scheduler, so
          // dependent chains, not issue slots, set its pace.
          auto pass_mask = [&](const uint32_t (&v)[32], int c) -> uint32_t {
            const int lim = n_valid - c * 32;  // columns >= lim are padding
            // Fast reject: with warm thresholds almost no chunk holds a passing score, and whether one does costs half the
            // instructions of locating it — the largest score of the chunk (3-input max tree), or with column scales the
            // smallest thr_s - v * cs (the same FFMA as the mask below, so the two can never disagree), then one vote.
            if (lim >= 32) {  // warp-uniform
              bool hit;
              if (has_scale) {
                float dmin = INFINITY;
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                  const float4 ca = *reinterpret_cast<const float4*>(cs_smem + c * 32 + 8 * g);
                  const float4 cb4 = *reinterpret_cast<const float4*>(cs_smem + c * 32 + 8 * g + 4);
                  const float d0 = fmaf(-__uint_as_float(v[8 * g + 0]), ca.x, thr_s);
                  const float d1 = fmaf(-__uint_as_float(v[8 * g + 1]), ca.y, thr_s);
                  const float d2 = fmaf(-__uint_as_float(v[8 * g + 2]), ca.z, thr_s);
                  const float d3 = fmaf(-__uint_as_float(v[8 * g + 3]), ca.w, thr_s);
                  const float d4 = fmaf(-__uint_as_float(v[8 * g + 4]), cb4.x, thr_s);
                  const float d5 = fmaf(-__uint_as_float(v[8 * g + 5]), cb4.y, thr_s);
                  const float d6 = fmaf(-__uint_as_float(v[8 * g + 6]), cb4.z, thr_s);
                  const float d7 = fmaf(-__uint_as_float(v[8 * g + 7]), cb4.w, thr_s);
                  dmin = fminf(fminf(dmin, fminf(fminf(d0, d1), d2)), fminf(fminf(fminf(d3, d4), d5), fminf(d6, d7)));
                }
                hit = dmin < 0.0f;
              } else {
                float vmax = -INFINITY;
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                  vmax = fmaxf(fmaxf(vmax, fmaxf(__uint_as_float(v[j]), __uint_as_float(v[j + 1]))),
                               fmaxf(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])));
                hit = vmax > thr;
              }
              if (!__any_sync(full, hit)) return 0u;
            }
            uint32_t mq[4] = {0u, 0u, 0u, 0u};
            if (has_scale) {  // warp-uniform: two straight-line bodies, not per-score predication
#pragma unroll
              for (int t = 7; t >= 0; --t) {
#pragma unroll
                for (int qd = 0; qd < 4; ++qd) {
                  const int j = qd * 8 + t;
                  const float dlt = fmaf(-__uint_as_float(v[j]), cs_smem[c * 32 + j], thr_s);
                  mq[qd] = __funnelshift_l(__float_as_uint(dlt), mq[qd], 1);  // mq = mq << 1 | sign(dlt)
                }
              }
            } else {
#pragma unroll
              for (int t = 7; t >= 0; --t) {
#pragma unroll
                for (int qd = 0; qd < 4; ++qd) {
                  const int j = qd * 8 + t;
                  const float dlt = thr - __uint_as_float(v[j]);
                  mq[qd] = __funnelshift_l(__float_as_uint(dlt), mq[qd], 1);
                }
              }
            }
            const uint32_t m = mq[0] | (mq[1] << 8) | (mq[2] << 16) | (mq[3] << 24);
            return lim >= 32 ? m : (m & ((1u << lim) - 1u));
          };
          auto append_and_cut = [&](const uint32_t (&v)[32], uint32_t m, int c) {
            // Each lane walks its OWN hits (the loop runs max-over-lanes popc(m) times, usually 0..2) and fetches v[j]
            // with a branch-free 5-level select tree, since registers cannot be indexed dynamically.  (Walking the union
            // of the lanes' hit columns with a warp-uniform switch was measured 25-75% slower: more iterations, and a
            // branch tree instead of selects.)  A filtered search drops the disallowed documents here, after the fast reject
            // and before anything is listed or cut, so no list cut or threshold is ever set by a document the query may
            // not return (with column scales the mask is conservative either way: the exact re-check below still runs).
            // The query's `allow` row is looked up here, on the rare append path, rather than held in a register for the
            // whole unit: that register costs the unfiltered WIDE kernels extra spills (ptxas -v).
            if (p.filter.on && m) m &= filter_mask32(p.filter, filter_row(p.filter, row), cb + c * 32);
            while (m) {
              const int j = __ffs(m) - 1;
              m &= m - 1;
              const uint32_t x = select32(v, j);
              float sc = __uint_as_float(x);
              if (has_scale) {
                sc *= (qs * cs_smem[c * 32 + j]);
                if (!(sc > thr)) continue;  // the folded filter is conservative: exact re-check
              }
              st_cg_u64(buf + cnt, make_key(f32_to_key(sc), uint32_t(cb + c * 32 + j)));
              ++cnt;
            }
            // keep >= 32 free slots for the next chunk; cut full lists back to their top-k
            uint32_t need = __ballot_sync(full, cnt + 32u > uint32_t(p.cap));
            while (need) {
              const int r = __ffs(need) - 1;
              need &= need - 1;
              const int n_r = __shfl_sync(full, int(cnt), r);
              const int64_t row_r = int64_t(m_tile) * BM + quarter * 32 + r;
              uint64_t* buf_r = p.cand + (int64_t(list_idx) * p.row_pad + row_r) * p.cap;
              const uint32_t vk = warp_compact_topk(buf_r, n_r, p.k, hist, list_stage, kListEntries, lane);
              if (lane == r) {
                cnt = uint32_t(p.k);
                thr_local = key_to_f32(vk);
                thr = fmaxf(thr, thr_local);
                atomicMax(p.gthr + row, vk);  // publish: valid lower bound of this query's global k-th score
              }
            }
          };
          uint32_t va[32], vb[32];
          tmem_ld_32x32(t_addr, va);
#pragma unroll 1
          for (int c = 0; c < nchunks; c += 2) {
            const bool has_b = c + 1 < nchunks;
            tmem_ld_wait();
            if (has_b) tmem_ld_32x32(t_addr + uint32_t((c + 1) * 32), vb);
            const uint32_t ma = pass_mask(va, c);
            if (has_b) tmem_ld_wait();  // vb is architecturally complete before any store / call below
            append_and_cut(va, ma, c);
            if (has_b) {
              const bool has_a2 = c + 2 < nchunks;
              if (has_a2) tmem_ld_32x32(t_addr + uint32_t((c + 2) * 32), va);
              const uint32_t mb = pass_mask(vb, c + 1);
              if (has_a2) tmem_ld_wait();
              append_and_cut(vb, mb, c + 1);
            }
          }
        } else {
#pragma unroll 1
          for (int c = 0; c < BN / 32; ++c) {
            if (c * 32 >= n_valid) break;  // warp-uniform
            uint32_t v[32];
            tmem_ld_32x32(t_addr + uint32_t(c * 32), v);
            tmem_ld_wait();
            const int col_lim = n_valid - c * 32;  // columns >= col_lim are padding
            if (EPI == EPI_STORE) {
              if (row_valid) {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (j < col_lim) p.dbg_scores[row * p.cols + cb + c * 32 + j] = __uint_as_float(v[j]);
              }
            } else {  // EPI_MAXTOK
              const int64_t base = cb + c * 32;
              const int64_t tok = base + lane;
              const bool mval = (tok < c1) && (p.mask == nullptr || p.mask[tok] != 0);
              uint32_t m = __ballot_sync(full, mval);  // valid tokens of the chunk still to be folded
              const int ncols = col_lim < 32 ? col_lim : 32;
              // Usually no document ends inside the chunk: one pass over its 32 columns.  When one does, the columns before
              // the end are folded, the document is emitted, and the pass repeats over the rest (the loop body exists once:
              // the kernel's instruction footprint matters more than the second pass).
#pragma unroll 1
              for (;;) {
                const int64_t lim = seg_end - base;  // columns of the chunk that belong to the current document
                const bool ends_here = lim < int64_t(ncols);  // warp-uniform
                const uint32_t part = ends_here ? (m & ((1u << int(lim)) - 1u)) : m;
                if (part) {
#pragma unroll
                  for (int j = 0; j < 32; ++j)
                    if ((part >> j) & 1u) run_max = fmaxf(run_max, __uint_as_float(v[j]) + bias_v);
                }
                if (!ends_here) break;
                m &= ~part;
                emit_doc();
                if (p.cu_seqlens) {
                  seg_end = next_end;
                  next_end = p.cu_seqlens[min(seg + 2, p.n_segs)];
                } else {
                  seg_end += p.seg_len;
                }
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR && cta_rank != 0) mbar_arrive_cluster(mapa_cluster(tempty_bar(acc), 0));  // leader's barrier
          else mbar_arrive(tempty_bar(acc));
        }
        if (WIDE) {
          acc_phase ^= 1u;  // this set's buffer is reused every second tile
        } else if (++acc == ACC_STAGES) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
      if (EPI == EPI_TOPK && tile_valid) p.counts[int64_t(list_idx) * p.row_pad + row] = row_valid ? int32_t(cnt) : 0;
      if (EPI == EPI_MAXTOK && p.cu_seqlens == nullptr) {
        // the document the split ends with
        for (; seg < seg_stop;) emit_doc();
      }
      if (EPI == EPI_MAXTOK && p.cu_seqlens != nullptr && tile_valid) {
        // documents that end exactly where the split ends (and empty ones there) are this unit's; one that goes on is a piece
        while (seg < p.n_segs && seg_end <= c1) {
          emit_doc();
          seg_end = next_end;
          next_end = p.cu_seqlens[min(seg + 2, p.n_segs)];
        }
        float tail_piece = BF16_LOWEST;
        if (seg < p.n_segs) {  // the current document continues in the next split
          if (head_open) head_piece = run_max;  // ... and began before this one: a single piece
          else tail_piece = run_max;
        }
        if (row_valid) {
          p.edge[(int64_t(split) * 2 + 0) * p.rows + row] = head_piece;
          p.edge[(int64_t(split) * 2 + 1) * p.rows + row] = tail_piece;
        }
      }
    });
  }

  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();  // no CTA leaves while a peer can still multicast into it or signal its barriers
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------ host helpers
inline PFN_cuTensorMapEncodeTiled get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
  });
  return fn;
}

// 2-D bf16 row-major [rows, cols_used] with row pitch ld elements; box = [64 cols, box_rows], 128B swizzle.
inline int make_tmap(CUtensorMap* map, const void* base, int64_t rows, int64_t cols_used, int64_t ld, int box_rows) {
  auto fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return LR_ECUDA;
  }
  cuuint64_t gdim[2] = {cuuint64_t(cols_used), cuuint64_t(rows)};
  cuuint64_t gstr[1] = {cuuint64_t(ld) * 2};
  cuuint32_t box[2] = {cuuint32_t(BK), cuuint32_t(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)", int(r),
              (long long)rows, (long long)cols_used, (long long)ld);
    return LR_ECUDA;
  }
  return LR_OK;
}

// balanced bands of row tiles: every band but the last holds band_size tiles
inline void plan_bands(int m_tiles, int band_max, int& band_size, int& n_bands) {
  if (band_max < 1) band_max = 1;
  n_bands = (m_tiles + band_max - 1) / band_max;
  if (n_bands < 1) n_bands = 1;
  band_size = (m_tiles + n_bands - 1) / n_bands;
  if (band_size < 1) band_size = 1;
  n_bands = (m_tiles + band_size - 1) / band_size;
}

template <int EPI, int CL, bool PAIR = false, bool BIGLIST = false, bool WIDE = false>
inline int launch_umma_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& prm, int grid,
                            cudaStream_t st) {
  auto kern = umma_gemm_kernel<EPI, CL, PAIR, BIGLIST, WIDE>;
  int rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), GEMM_SMEM_TOTAL);
  if (rc) return rc;
  cudaError_t e;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned(grid));
  cfg.blockDim = dim3(WIDE ? GEMM_THREADS_WIDE : GEMM_THREADS);
  cfg.dynamicSmemBytes = GEMM_SMEM_TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // The team schedule only pays when the whole grid is co-resident (one cluster per SM pair).  On a device where fewer
  // clusters fit (a smaller part, MPS with an SM limit) the same units are walked round robin instead: the unit set
  // (row group x split) and the candidate-list layout do not depend on the schedule.
  GemmParams prm_rr;
  const GemmParams* pp = &prm;
  if (prm.sched != 0) {
    static int max_clusters[64];  // per device, this kernel instance; 0 = not queried yet
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64) {
      if (max_clusters[dev] == 0) {
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n <= 0) {
          cudaGetLastError();
          n = -1;  // unknown: trust the plan (the in-kernel wait is bounded either way)
        }
        max_clusters[dev] = n;
      }
      if (max_clusters[dev] > 0 && max_clusters[dev] * CL < grid) {
        prm_rr = prm;
        prm_rr.sched = 0;
        pp = &prm_rr;
      }
    }
  }
  ProfileEvents& pe = profile_events();
  if (pe.begin && pe.end) LR_CUDA(cudaEventRecord(pe.begin, st));
  e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, *pp);
  if (e != cudaSuccess) {
    set_error("kernel launch failed: %s (grid=%d cluster=%d)", cudaGetErrorString(e), grid, CL);
    return LR_ECUDA;
  }
  count_launch();
  if (pe.begin && pe.end) LR_CUDA(cudaEventRecord(pe.end, st));
  return LR_OK;
}

// Work plan shared by the hosts of K2 and K3: groups of CL row tiles, bands of groups, grid of whole clusters.
struct GemmGeometry {
  int cl, pair, m_tiles, m_groups, band_size, n_bands, n_clusters;
};
// mode: 0 = auto, 1 = single CTA, 2 = cluster of 2 with multicast B, 3 = cta_group::2 pair
inline GemmGeometry plan_geometry(int64_t rows, int band_max_tiles, int mode) {
  GemmGeometry g{};
  g.m_tiles = int((rows + BM - 1) / BM);
  g.cl = (g.m_tiles >= 2) ? 2 : 1;
  g.pair = 0;
  if (mode == 1) g.cl = 1;
  if (mode == 2) g.cl = 2;
  if (mode == 3) { g.cl = 2; g.pair = 1; }
  g.m_groups = (g.m_tiles + g.cl - 1) / g.cl;
  int band_max = band_max_tiles / g.cl;
  plan_bands(g.m_groups, band_max < 1 ? 1 : band_max, g.band_size, g.n_bands);
  g.n_clusters = sm_count() / g.cl;
  if (g.n_clusters < 1) g.n_clusters = 1;
  return g;
}

// Team schedule for a fixed number of splits: the band width g (row groups per band) that keeps the most clusters busy
// when each band's floor(nc / g) teams share `splits` splits.  Returns 0 when no width reaches `min_util`.
inline int plan_team_band(int m_groups, int nc, int splits, double min_util, int g_max = 20) {
  double best = min_util;
  int best_g = 0;
  const int g_hi = m_groups < g_max ? m_groups : g_max;
  for (int g = (m_groups < 4 ? m_groups : 4); g <= g_hi && g <= nc; ++g) {
    const int q = m_groups / g, r = m_groups % g;
    const int n_main = nc / g, n_rem = r ? nc / r : 0;
    const int64_t time = int64_t(q) * ((splits + n_main - 1) / n_main) + (r ? (splits + n_rem - 1) / n_rem : 0);
    const double util = double(m_groups) * splits / (double(nc) * double(time));
    const double score = util - 0.0005 * (q + (r ? 1 : 0));  // ties: fewer passes over the column operand
    if (score > best) {
      best = score;
      best_g = g;
    }
  }
  return best_g;
}

}  // namespace lr
