// sparse_head.cu — K3: document sparse head.
//
//   lr_sparse_head_max     out[b, v] = log1p(relu(max_{t valid} (h[b,t,:] . W[v,:] + bias[v])))
//       replaces aggregate()/max_linear_mapping  (reference finetune/sparse_pooling.py:244-278,
//       utils/max_linear_map.py:10-90: a Python loop over seq positions, one GEMM + 4 elementwise launches
//       per token) and relu_/log1p_ (finetune/modeling_hybrid.py:183-187).
//       One umma_gemm_kernel<EPI_MAXTOK> launch: rows = vocabulary (A = lm_head.weight [V, d]), columns = tokens
//       (B = hidden [B*S, d]); the per-token logits never leave TMEM/registers.
//   lr_sparsify_quantize   top_k_sampling (finetune/sparse_pooling.py:89-106) + the quantiser of
//       convert_sparse_reps_to_json_pt (finetune/sparse_converter_mixin.py:103-160) -> CSR (indptr, tok, impact).
#include "umma_gemm.cuh"

namespace lr {

constexpr int SP_THREADS = 256;

// ---- per document: threshold = k_eff-th largest value (radix select over f32 keys), count of surviving non-zeros
__global__ void __launch_bounds__(SP_THREADS)
sparsify_select_kernel(const float* __restrict__ reps, int64_t V, int k_eff, float quant, float* thr_out,
                       int32_t* cnt_out) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t s_bin, s_remaining;
  __shared__ int s_cnt;
  const int64_t b = blockIdx.x;
  const float* x = reps + b * V;
  const int tid = threadIdx.x;
  uint32_t thr_key = 0;  // keep everything
  if (k_eff > 0) {
    uint32_t prefix = 0, remaining = uint32_t(k_eff);
    for (int pass = 3; pass >= 0; --pass) {
      const int shift = pass * 8;
      hist[tid] = 0;
      __syncthreads();
      for (int64_t i = tid; i < V; i += SP_THREADS) {
        const uint32_t h = f32_to_key(x[i]);
        if (pass == 3 || (h >> (shift + 8)) == prefix) atomicAdd(&hist[(h >> shift) & 0xFFu], 1u);
      }
      __syncthreads();
      if (tid < 32) {
        const int base = 8 * (31 - tid);
        uint32_t c[8], sum = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          c[i] = hist[base + 7 - i];
          sum += c[i];
        }
        uint32_t incl = sum;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, off);
          if (tid >= off) incl += t;
        }
        const uint32_t excl = incl - sum;
        if (excl < remaining && remaining <= incl) {
          uint32_t acc = excl;
          bool done = false;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (!done && acc + c[i] >= remaining) {
              s_bin = uint32_t(base + 7 - i);
              s_remaining = remaining - acc;
              done = true;
            }
            if (!done) acc += c[i];
          }
        }
      }
      __syncthreads();
      prefix = (prefix << 8) | s_bin;
      remaining = s_remaining;
      __syncthreads();
    }
    thr_key = prefix;
  }
  const float thr = k_eff > 0 ? key_to_f32(thr_key) : -INFINITY;
  // torch: indices_to_remove = scores < kth  ->  keep x >= thr (all ties kept)
  if (tid == 0) s_cnt = 0;
  __syncthreads();
  int local = 0;
  for (int64_t i = tid; i < V; i += SP_THREADS) {
    const float v = x[i];
    if (v >= thr) {
      const float qv = rintf(fmaxf(v, 0.0f) * quant);  // torch.round = round half to even
      if (qv >= 1.0f) ++local;
    }
  }
  if (local) atomicAdd(&s_cnt, local);
  __syncthreads();
  if (tid == 0) {
    thr_out[b] = thr;
    cnt_out[b] = s_cnt;
  }
}

__global__ void exclusive_scan_kernel(const int32_t* cnt, int64_t B, int32_t* indptr) {
  // single thread block, sequential over chunks (B is a batch size)
  if (threadIdx.x == 0) {
    long long run = 0;
    for (int64_t b = 0; b < B; ++b) {
      indptr[b] = int32_t(run);
      run += cnt[b];
    }
    indptr[B] = int32_t(run);
  }
}

// cu[0] = 0, cu[b] = lens[0] + ... + lens[b-1] where lens[b] arrives in cu[b + 1] (B is a batch size: one thread)
__global__ void inclusive_scan_kernel(int32_t* cu, int64_t B) {
  if (threadIdx.x == 0) {
    int32_t run = 0;
    cu[0] = 0;
    for (int64_t b = 1; b <= B; ++b) {
      run += cu[b];
      cu[b] = run;
    }
  }
}

// ---- per document: ordered write of (token id, impact)
__global__ void __launch_bounds__(SP_THREADS)
sparsify_write_kernel(const float* __restrict__ reps, int64_t V, float quant, const float* thr_in,
                      const int32_t* __restrict__ indptr, int32_t* tok, uint16_t* impact, int64_t cap) {
  __shared__ int warp_tot[SP_THREADS / 32];
  __shared__ int s_base;
  const int64_t b = blockIdx.x;
  const float* x = reps + b * V;
  const float thr = thr_in[b];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_base = indptr[b];
  __syncthreads();
  for (int64_t i0 = 0; i0 < V; i0 += SP_THREADS) {
    const int64_t i = i0 + tid;
    float qv = 0.0f;
    if (i < V) {
      const float v = x[i];
      if (v >= thr) qv = rintf(fmaxf(v, 0.0f) * quant);
    }
    const bool keep = qv >= 1.0f;
    const uint32_t m = __ballot_sync(0xFFFFFFFFu, keep);
    if (lane == 0) warp_tot[warp] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < SP_THREADS / 32; ++w) {
      const int t = warp_tot[w];
      if (w < warp) before += t;
      total += t;
    }
    const int base = s_base;
    if (keep) {
      const int64_t pos = int64_t(base) + before + __popc(m & ((1u << lane) - 1u));
      if (pos < cap) {
        tok[pos] = int32_t(i);
        impact[pos] = uint16_t(fminf(qv, 65535.0f));
      }
    }
    __syncthreads();
    if (tid == 0) s_base = base + total;
    __syncthreads();
  }
}

// ---- top_p_sampling (finetune/sparse_pooling.py:64-87): ascending sort, softmax, cumulative sum; an entry is zeroed while
// the cumulative probability up to and including it is <= 1 - top_p, and the last min_keep entries of the sorted order
// (the largest) always stay.  Here without a sort: an 8-bit radix descent over the order-preserving keys finds the
// value at which the cumulative mass crosses 1 - top_p (masses as 2^-44 fixed point in u64, so the sums do not depend on
// the order of the atomics); entries below it go, and of the entries equal to it the first few by index (a stable
// sort's order).  One CTA per document; in place.
constexpr int TP_THREADS = 512;
constexpr double TP_SCALE = 17592186044416.0;  // 2^44

__device__ __forceinline__ float tp_block_max(float v, float* red) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) v = fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, off));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
  for (int i = 1; i < TP_THREADS / 32; ++i) r = fmaxf(r, red[i]);
  return r;
}

__global__ void __launch_bounds__(TP_THREADS)
top_p_filter_kernel(float* __restrict__ reps, int64_t V, float top_p, int min_keep) {
  __shared__ unsigned long long mass[256];
  __shared__ uint32_t cnt[256];
  __shared__ float red[TP_THREADS / 32];
  __shared__ double red_d[TP_THREADS / 32];
  __shared__ uint32_t s_bin, s_below_cnt, s_eq;
  __shared__ unsigned long long s_below_mass;
  __shared__ uint32_t s_tie_seen;
  float* x = reps + int64_t(blockIdx.x) * V;
  const int tid = threadIdx.x;
  // softmax denominator (double: the reference accumulates 1e5 float terms; no order of ours reproduces its rounding)
  float mx = -INFINITY;
  for (int64_t i = tid; i < V; i += TP_THREADS) mx = fmaxf(mx, x[i]);
  mx = tp_block_max(mx, red);
  double z = 0.0;
  for (int64_t i = tid; i < V; i += TP_THREADS) z += double(expf(x[i] - mx));
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) z += __shfl_xor_sync(0xFFFFFFFFu, z, off);
  if ((tid & 31) == 0) red_d[tid >> 5] = z;
  __syncthreads();
  z = 0.0;
  for (int i = 0; i < TP_THREADS / 32; ++i) z += red_d[i];
  const double inv_z = TP_SCALE / z;
  auto mass_of = [&](float v) { return static_cast<unsigned long long>(double(expf(v - mx)) * inv_z + 0.5); };
  // cumulative mass that may be removed; the count cap keeps the min_keep largest
  const unsigned long long target = static_cast<unsigned long long>((1.0 - double(top_p)) * TP_SCALE);
  const uint32_t max_remove = V > min_keep ? uint32_t(V - min_keep) : 0u;
  // ---- descent 1: by mass.  prefix = key bits fixed so far; below = (mass, count) of all keys smaller than the prefix range
  uint32_t prefix = 0;
  unsigned long long below_mass = 0;
  uint32_t below_cnt = 0;
  for (int pass = 3; pass >= 0; --pass) {
    const int shift = pass * 8;
    if (tid < 256) {
      mass[tid] = 0;
      cnt[tid] = 0;
    }
    __syncthreads();
    for (int64_t i = tid; i < V; i += TP_THREADS) {
      const uint32_t k = f32_to_key(x[i]);
      if (pass == 3 || (k >> (shift + 8)) == prefix) {
        atomicAdd(&mass[(k >> shift) & 0xFFu], mass_of(x[i]));
        atomicAdd(&cnt[(k >> shift) & 0xFFu], 1u);
      }
    }
    __syncthreads();
    if (tid == 0) {  // ascending walk: the first bin whose cumulative mass exceeds the target holds the crossing value
      unsigned long long m = below_mass;
      uint32_t c = below_cnt;
      int b = 0;
      for (; b < 255; ++b) {
        if (m + mass[b] > target) break;
        m += mass[b];
        c += cnt[b];
      }
      s_bin = uint32_t(b);
      s_below_mass = m;
      s_below_cnt = c;
      s_eq = cnt[b];  // after the last pass: the number of entries equal to the crossing value
    }
    __syncthreads();
    prefix = (prefix << 8) | s_bin;
    below_mass = s_below_mass;
    below_cnt = s_below_cnt;
    __syncthreads();
  }
  // entries with a smaller key go; of the s_eq entries equal to it, the first `ties` by index
  uint32_t vkey = prefix;
  uint32_t ties;
  {
    const unsigned long long mv = mass_of(key_to_f32(vkey));
    // zero-mass entries never move the sum: all of them are at or below the bound
    const unsigned long long t = mv == 0 ? 0xFFFFFFFFull : (target >= below_mass ? (target - below_mass) / mv : 0ull);
    ties = t > s_eq ? s_eq : uint32_t(t);
  }
  if (below_cnt + ties > max_remove) {
    // ---- descent 2: the min_keep cap binds: remove exactly the max_remove smallest, i.e. cut at that rank's value
    uint32_t pre2 = 0, below2 = 0;
    for (int pass = 3; pass >= 0; --pass) {
      const int shift = pass * 8;
      if (tid < 256) cnt[tid] = 0;
      __syncthreads();
      for (int64_t i = tid; i < V; i += TP_THREADS) {
        const uint32_t k = f32_to_key(x[i]);
        if (pass == 3 || (k >> (shift + 8)) == pre2) atomicAdd(&cnt[(k >> shift) & 0xFFu], 1u);
      }
      __syncthreads();
      if (tid == 0) {
        uint32_t c = below2;
        int b = 0;
        for (; b < 255; ++b) {
          if (c + cnt[b] > max_remove) break;
          c += cnt[b];
        }
        s_bin = uint32_t(b);
        s_below_cnt = c;
      }
      __syncthreads();
      pre2 = (pre2 << 8) | s_bin;
      below2 = s_below_cnt;
      __syncthreads();
    }
    vkey = pre2;
    ties = max_remove - below2;
  }
  // ---- apply: ties are taken in index order (chunks of the block, ballot scan inside a chunk)
  if (tid == 0) s_tie_seen = 0;
  __syncthreads();
  __shared__ uint32_t warp_eq[TP_THREADS / 32];
  for (int64_t i0 = 0; i0 < V; i0 += TP_THREADS) {
    const int64_t i = i0 + tid;
    const uint32_t k = i < V ? f32_to_key(x[i]) : 0xFFFFFFFFu;
    const bool eq = i < V && k == vkey;
    const uint32_t em = __ballot_sync(0xFFFFFFFFu, eq);
    if ((tid & 31) == 0) warp_eq[tid >> 5] = __popc(em);
    __syncthreads();
    uint32_t before = s_tie_seen, total = 0;
    for (int w = 0; w < TP_THREADS / 32; ++w) {
      if (w < (tid >> 5)) before += warp_eq[w];
      total += warp_eq[w];
    }
    const uint32_t rank = before + __popc(em & ((1u << (tid & 31)) - 1u));
    if (i < V && (k < vkey || (eq && rank < ties))) x[i] = 0.0f;
    __syncthreads();
    if (tid == 0) s_tie_seen += total;
    __syncthreads();
  }
}

// ---- packed tokens: documents that cross a split boundary
// tiles [t0, t1) of split s (the same balanced ranges as umma_gemm.cuh split_cols)
__device__ __forceinline__ void packed_split_range(int split, int splits, int64_t n_tiles, int64_t T, int64_t& c0, int64_t& c1) {
  c0 = (int64_t(split) * n_tiles) / splits * BN;
  c1 = (int64_t(split + 1) * n_tiles) / splits * BN;
  if (c1 > T) c1 = T;
}

// split_doc0[s] = document holding the first token of split s (the first one that ends after it); 0 for split 0, whose
// unit also emits the empty documents the batch may begin with
__global__ void split_doc0_kernel(const int32_t* __restrict__ cu, int64_t B, int64_t T, int64_t n_tiles, int splits,
                                  int32_t* split_doc0) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= splits) return;
  int64_t c0, c1;
  packed_split_range(s, splits, n_tiles, T, c0, c1);
  int64_t lo = 0, hi = B - 1;  // smallest d with cu[d + 1] > c0
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (int64_t(cu[mid + 1]) > c0) hi = mid; else lo = mid + 1;
  }
  split_doc0[s] = s == 0 ? 0 : int32_t(lo);
}

// grid (splits - 1, row chunks): boundary b lies between split b - 1 and split b.  A document that crosses it was left
// in pieces (GemmParams::edge); the CTA of the FIRST boundary a document crosses combines all of them.
__global__ void __launch_bounds__(256)
sparse_head_fix_kernel(const int32_t* __restrict__ cu, const int32_t* __restrict__ split_doc0, const float* __restrict__ edge,
                       int64_t rows, int64_t B, int64_t T, int64_t n_tiles, int splits, int relu, int log1p, float* out) {
  const int b = blockIdx.x + 1;
  int64_t c0, c1, p0, p1;
  packed_split_range(b, splits, n_tiles, T, c0, c1);
  packed_split_range(b - 1, splits, n_tiles, T, p0, p1);
  const int64_t d = split_doc0[b];
  const int64_t d_begin = cu[d], d_end = cu[d + 1];
  if (d_begin >= c0) return;            // the document starts at the boundary: nothing crosses
  if (b > 1 && d_begin < p0) return;    // it crossed an earlier boundary: that CTA's work
  (void)B;
  for (int64_t row = int64_t(blockIdx.y) * blockDim.x + threadIdx.x; row < rows; row += int64_t(gridDim.y) * blockDim.x) {
    float acc = edge[(int64_t(b - 1) * 2 + 1) * rows + row];
    for (int s = b; s < splits; ++s) {
      acc = fmaxf(acc, edge[(int64_t(s) * 2 + 0) * rows + row]);
      int64_t s0, s1;
      packed_split_range(s, splits, n_tiles, T, s0, s1);
      if (d_end <= s1) break;
    }
    float x = acc;
    if (relu) x = fmaxf(x, 0.0f);
    if (log1p) x = log1pf(x);
    out[d * rows + row] = x;
  }
}

// ---- packing: the valid tokens of every document, concatenated (what the packed GEMM multiplies)
__global__ void __launch_bounds__(256) pack_count_kernel(const uint8_t* __restrict__ mask, int64_t S, int32_t* lens) {
  __shared__ int s_tot;
  const int64_t b = blockIdx.x;
  if (threadIdx.x == 0) s_tot = 0;
  __syncthreads();
  int local = 0;
  for (int64_t t = threadIdx.x; t < S; t += blockDim.x) local += mask[b * S + t] != 0;
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) local += __shfl_xor_sync(0xFFFFFFFFu, local, off);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(&s_tot, local);
  __syncthreads();
  if (threadIdx.x == 0) lens[b] = s_tot;
}

// grid (B, PACK_SLICES): every CTA ranks the valid tokens of its document (warp 0, ballot scan) and its warps copy the
// rows of one slice of the document, 16 bytes per lane
constexpr int PACK_SLICES = 4;
__global__ void __launch_bounds__(256) pack_rows_kernel(const uint8_t* __restrict__ hidden, const uint8_t* __restrict__ mask,
                                                        int64_t S, int64_t row_bytes, const int32_t* __restrict__ cu_seqlens,
                                                        uint8_t* __restrict__ packed, int64_t cap) {
  extern __shared__ int32_t pk_pos[];  // [S]: destination row inside the document, -1 for masked tokens
  const int64_t b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    int run = 0;
    for (int64_t t0 = 0; t0 < S; t0 += 32) {
      const int64_t t = t0 + lane;
      const bool v = t < S && mask[b * S + t] != 0;
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, v);
      if (t < S) pk_pos[t] = v ? run + __popc(m & ((1u << lane) - 1u)) : -1;
      run += __popc(m);
    }
  }
  __syncthreads();
  const int64_t base = cu_seqlens[b];
  const int64_t per = (S + PACK_SLICES - 1) / PACK_SLICES;
  const int64_t t_lo = int64_t(blockIdx.y) * per, t_hi = min(S, t_lo + per);
  for (int64_t t = t_lo + warp; t < t_hi; t += blockDim.x / 32) {
    const int pos = pk_pos[t];
    if (pos < 0 || base + pos >= cap) continue;
    const uint4* src = reinterpret_cast<const uint4*>(hidden + (b * S + t) * row_bytes);
    uint4* dst = reinterpret_cast<uint4*>(packed + (base + pos) * row_bytes);
    for (int64_t i = lane; i < row_bytes / 16; i += 32) dst[i] = ld_nc_v4(src + i);
  }
}

}  // namespace lr

using namespace lr;

// Packed tokens: splits = balanced ranges of whole tiles, ~2 tiles each and at most 64 of them (the edge buffer holds two
// rows of V floats per split).
struct PackedPlan {
  int64_t n_tiles;
  int splits;
  size_t off_doc0, off_edge, total_bytes;  // workspace: team counters | split_doc0 | edge
};
static PackedPlan packed_plan(int64_t T, int64_t V) {
  PackedPlan pp{};
  pp.n_tiles = (T + BN - 1) / BN;
  int64_t tps = (pp.n_tiles + 63) / 64;
  if (tps < 2) tps = 2;
  const int forced_tps = knobs().head_tiles_per_split;  // tests: 1 = a cut every 256 tokens
  if (forced_tps != KNOB_UNSET) tps = forced_tps;
  if (tps < 1) tps = 1;
  int64_t splits = (pp.n_tiles + tps - 1) / tps;
  if (splits < 1) splits = 1;
  pp.splits = int(splits);
  pp.off_doc0 = 64 * 1024;  // team progress counters: n_bands * n_clusters words (<= 126 * 74)
  pp.off_edge = pp.off_doc0 + ((size_t(pp.splits) * 4 + 255) / 256) * 256;
  pp.total_bytes = pp.off_edge + size_t(pp.splits) * 2 * size_t(V) * 4;
  return pp;
}

// cols = token rows of `hidden`; documents are seg_len tokens each (cu_seqlens == null) or the packed runs cu_seqlens
// describes (mask == null then: every packed token is valid; `ws` = workspace of packed_plan())
static int sparse_head_launch(const void* hidden, const void* W, const float* bias, const uint8_t* mask,
                              const int32_t* cu_seqlens, int64_t B, int64_t S, int64_t cols, int64_t d, int64_t V, int relu,
                              int log1p, float* out, uint8_t* ws, cudaStream_t st) {
  CUtensorMap tmA, tmB;
  int rc;
  int sps = 1, splits;
  PackedPlan pp{};
  const Knobs& kn = knobs();
  if (cu_seqlens) {
    pp = packed_plan(cols, V);
    splits = pp.splits;
  } else {
    // a unit covers whole documents and at least ~2 column tiles
    sps = int((2 * BN + S - 1) / S);
    if (sps < 1) sps = 1;
    if (kn.head_docs_per_unit != KNOB_UNSET) sps = kn.head_docs_per_unit;
    if (sps > B) sps = int(B);
    splits = int((B + sps - 1) / sps);
  }
  // Vocabulary bands x document splits.  With enough of both, fixed teams of clusters walk the splits of a band in step
  // (umma_gemm.cuh for_each_unit): a hidden-state tile is fetched from HBM once per team and the band's lm_head rows
  // stay L2-resident; the team schedule runs as cta_group::2 pairs.  Otherwise round robin over 12-tile bands.
  int mode = kn.head_cluster;
  int team_band = 0;
  if (kn.head_sched != 0 && mode != 1 && V > 8 * 2 * BM && splits >= 2) {
    const int m_groups = int((V + 2 * BM - 1) / (2 * BM));
    team_band = kn.head_team_band != KNOB_UNSET ? kn.head_team_band
                                                 : plan_team_band(m_groups, sm_count() / 2, splits, 0.85);
    if (team_band > m_groups) team_band = m_groups;
    if (team_band > 0 && mode == 0) mode = 3;
  }
  const GemmGeometry geo = plan_geometry(V, 12, mode);
  if ((rc = make_tmap(&tmA, W, V, d, d, BM))) return rc;
  if ((rc = make_tmap(&tmB, hidden, cols, d, d, BN / geo.cl))) return rc;
  GemmParams prm{};
  prm.rows = V; prm.cols = cols;
  prm.m_tiles = geo.m_tiles; prm.m_groups = geo.m_groups;
  prm.row_pad = int64_t(prm.m_tiles) * BM;
  prm.kblocks = int((d + BK - 1) / BK);
  prm.seg_len = S; prm.n_segs = B;
  prm.segs_per_split = sps;
  prm.splits = splits;
  if (cu_seqlens) {
    prm.cu_seqlens = cu_seqlens;
    prm.n_tiles = int(pp.n_tiles);
    prm.tile_begin = 0;
    prm.split_doc0 = reinterpret_cast<const int32_t*>(ws + pp.off_doc0);
    prm.edge = reinterpret_cast<float*>(ws + pp.off_edge);
    split_doc0_kernel<<<(splits + 127) / 128, 128, 0, st>>>(cu_seqlens, B, cols, pp.n_tiles, splits,
                                                          reinterpret_cast<int32_t*>(ws + pp.off_doc0));
    LR_LAUNCH_CHECK();
  }
  prm.band_size = geo.band_size; prm.n_bands = geo.n_bands;
  prm.units = prm.m_groups * prm.splits;
  prm.bias = bias; prm.mask = mask; prm.out = out; prm.relu = relu; prm.log1p = log1p;
  int clusters = prm.units < geo.n_clusters ? prm.units : geo.n_clusters;
  uint32_t* team_ctr = nullptr;
  bool own_ctr = false;
  if (team_band > 0 && geo.cl == 2) {
    prm.sched = 1;
    prm.team_window = kn.head_team_window;
    prm.band_size = team_band;
    prm.n_bands = (prm.m_groups + team_band - 1) / team_band;
    clusters = geo.n_clusters;
    // progress counters of the teams, one per (band, team): the head of the caller's workspace (packed entry point), or
    // stream-ordered scratch released after the launch
    const size_t ctr_bytes = size_t(prm.n_bands) * size_t(geo.n_clusters) * 4;
    if (ws && ctr_bytes <= pp.off_doc0) {
      team_ctr = reinterpret_cast<uint32_t*>(ws);
    } else {
      LR_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&team_ctr), ctr_bytes, st));
      own_ctr = true;
    }
    cudaError_t e = cudaMemsetAsync(team_ctr, 0, ctr_bytes, st);
    if (e != cudaSuccess) {
      if (own_ctr) cudaFreeAsync(team_ctr, st);
      set_error("sparse_head: cudaMemsetAsync failed: %s", cudaGetErrorString(e));
      return LR_ECUDA;
    }
    prm.team_ctr = team_ctr;
  }
  const int grid = clusters * geo.cl;
  if (geo.pair) rc = launch_umma_gemm<EPI_MAXTOK, 2, true>(tmA, tmB, prm, grid, st);
  else rc = geo.cl == 2 ? launch_umma_gemm<EPI_MAXTOK, 2>(tmA, tmB, prm, grid, st)
                        : launch_umma_gemm<EPI_MAXTOK, 1>(tmA, tmB, prm, grid, st);
  if (own_ctr) cudaFreeAsync(team_ctr, st);
  if (rc == LR_OK && cu_seqlens && splits > 1) {
    int chunks = int((V + 255) / 256);
    if (chunks > 64) chunks = 64;
    sparse_head_fix_kernel<<<dim3(unsigned(splits - 1), unsigned(chunks)), 256, 0, st>>>(
        cu_seqlens, prm.split_doc0, prm.edge, V, B, cols, pp.n_tiles, splits, relu, log1p, out);
    LR_LAUNCH_CHECK();
  }
  return rc;
}

extern "C" int lr_sparse_head_max(const void* hidden, const void* W, const float* bias, const uint8_t* mask,
                                  int64_t B, int64_t S, int64_t d, int64_t V, int relu, int log1p, float* out,
                                  void* stream) {
  LR_CHECK_ARG(hidden && W && mask && out, "sparse_head: null pointer");
  LR_CHECK_ARG(B >= 1 && S >= 1 && V >= 1, "sparse_head: B, S, V must be >= 1");
  LR_CHECK_ARG(d >= 8 && d % 8 == 0, "sparse_head: d (%lld) must be a positive multiple of 8", (long long)d);
  LR_CHECK_ARG((uintptr_t(hidden) & 15) == 0 && (uintptr_t(W) & 15) == 0, "sparse_head: hidden/W must be 16-byte aligned");
  LR_CHECK_ARG(B * S < (int64_t(1) << 31) - BN && V < (int64_t(1) << 31) - BM, "sparse_head: B*S or V too large");
  return sparse_head_launch(hidden, W, bias, mask, nullptr, B, S, B * S, d, V, relu, log1p, out, nullptr,
                            static_cast<cudaStream_t>(stream));
}

// Planner introspection (host only; CPU tests): out[4] = 256-token tiles, splits, edge-buffer offset, workspace bytes
extern "C" int lr_sparse_head_packed_plan(int64_t T, int64_t V, int64_t* out) {
  LR_CHECK_ARG(out && T >= 1 && V >= 1, "sparse_head_packed_plan: bad arguments");
  const PackedPlan pp = packed_plan(T, V);
  out[0] = pp.n_tiles; out[1] = pp.splits; out[2] = int64_t(pp.off_edge); out[3] = int64_t(pp.total_bytes);
  return LR_OK;
}

extern "C" size_t lr_sparse_head_packed_workspace_bytes(int64_t T, int64_t V) {
  if (T < 1 || V < 1) return 0;
  return packed_plan(T, V).total_bytes;
}

extern "C" int lr_sparse_head_max_packed(const void* hidden, const void* W, const float* bias, const int32_t* cu_seqlens,
                                         int64_t B, int64_t T, int64_t d, int64_t V, int relu, int log1p, float* out,
                                         void* workspace, size_t ws_bytes, void* stream) {
  LR_CHECK_ARG(hidden && W && cu_seqlens && out, "sparse_head_packed: null pointer");
  LR_CHECK_ARG(B >= 1 && T >= 1 && V >= 1, "sparse_head_packed: B, T, V must be >= 1");
  LR_CHECK_ARG(d >= 8 && d % 8 == 0, "sparse_head_packed: d (%lld) must be a positive multiple of 8", (long long)d);
  LR_CHECK_ARG((uintptr_t(hidden) & 15) == 0 && (uintptr_t(W) & 15) == 0, "sparse_head_packed: hidden/W must be 16-byte aligned");
  LR_CHECK_ARG(T < (int64_t(1) << 31) - BN && V < (int64_t(1) << 31) - BM, "sparse_head_packed: T or V too large");
  const size_t need = packed_plan(T, V).total_bytes;
  if (!workspace || ws_bytes < need || (uintptr_t(workspace) & 255)) {
    set_error("sparse_head_packed: workspace too small or misaligned (%zu given, %zu needed)", ws_bytes, need);
    return LR_EWORKSPACE;
  }
  return sparse_head_launch(hidden, W, bias, nullptr, cu_seqlens, B, 0, T, d, V, relu, log1p, out,
                            static_cast<uint8_t*>(workspace), static_cast<cudaStream_t>(stream));
}

extern "C" int lr_pack_tokens(const void* hidden, const uint8_t* mask, int64_t B, int64_t S, int64_t d, void* packed,
                              int64_t cap, int32_t* cu_seqlens, void* stream) {
  LR_CHECK_ARG(hidden && mask && packed && cu_seqlens, "pack_tokens: null pointer");
  LR_CHECK_ARG(B >= 1 && S >= 1 && d >= 8 && d % 8 == 0, "pack_tokens: bad sizes");
  LR_CHECK_ARG(B <= 65535 * 32 && S * 4 <= 200 * 1024, "pack_tokens: B or S too large");
  LR_CHECK_ARG((uintptr_t(hidden) & 15) == 0 && (uintptr_t(packed) & 15) == 0, "pack_tokens: buffers must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // lengths into cu_seqlens[1..B], then an in-place scan (cu_seqlens[0] = 0)
  pack_count_kernel<<<unsigned(B), 256, 0, st>>>(mask, S, cu_seqlens + 1);
  LR_LAUNCH_CHECK();
  inclusive_scan_kernel<<<1, 32, 0, st>>>(cu_seqlens, B);
  LR_LAUNCH_CHECK();
  int rc = ensure_dyn_smem(reinterpret_cast<const void*>(pack_rows_kernel), 200 * 1024);
  if (rc) return rc;
  pack_rows_kernel<<<dim3(unsigned(B), PACK_SLICES), 256, size_t(S) * 4, st>>>(
      static_cast<const uint8_t*>(hidden), mask, S, d * 2, cu_seqlens, static_cast<uint8_t*>(packed), cap);
  LR_LAUNCH_CHECK();
  return LR_OK;
}

extern "C" int lr_top_p_filter(float* reps, int64_t B, int64_t V, float top_p, int min_keep, void* stream) {
  LR_CHECK_ARG(reps, "top_p_filter: null pointer");
  LR_CHECK_ARG(B >= 1 && V >= 1 && V < (int64_t(1) << 31), "top_p_filter: bad sizes");
  LR_CHECK_ARG(min_keep >= 0, "top_p_filter: min_keep (%d) must be >= 0", min_keep);
  if (!(top_p > 0.0f && top_p < 1.0f)) return LR_OK;  // sparse_pooling.py:73-74: outside (0, 1) the filter is off
  // remove[..., -min_keep:] = False: with min_keep = 0 the slice -0: is every column, so nothing is removed
  if (min_keep == 0) return LR_OK;
  top_p_filter_kernel<<<unsigned(B), TP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(reps, V, top_p, min_keep);
  LR_LAUNCH_CHECK();
  return LR_OK;
}

extern "C" size_t lr_sparsify_scratch_bytes(int64_t B, int64_t V) {
  (void)V;
  return size_t(B > 0 ? B : 0) * 8 + 256;
}

extern "C" int lr_sparsify_quantize(const float* reps, int64_t B, int64_t V, int top_k, int min_keep, float quant,
                                    int32_t* indptr, int32_t* tok, uint16_t* impact, int64_t cap, void* scratch,
                                    void* stream) {
  LR_CHECK_ARG(reps && indptr && scratch, "sparsify: null pointer");
  LR_CHECK_ARG(B >= 1 && V >= 1 && V < (int64_t(1) << 31), "sparsify: bad sizes");
  LR_CHECK_ARG(cap >= 0 && (cap == 0 || (tok && impact)), "sparsify: null tok/impact");
  LR_CHECK_ARG(quant > 0.0f, "sparsify: quantization factor must be > 0");
  int k_eff = 0;  // top_k <= 0 disables the filter (sparse_pooling.py:98-99)
  if (top_k > 0) {
    k_eff = top_k > min_keep ? top_k : min_keep;
    if (k_eff > V) k_eff = int(V);
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* thr = static_cast<float*>(scratch);
  int32_t* cnt = reinterpret_cast<int32_t*>(thr + B);
  sparsify_select_kernel<<<unsigned(B), SP_THREADS, 0, st>>>(reps, V, k_eff, quant, thr, cnt);
  LR_LAUNCH_CHECK();
  exclusive_scan_kernel<<<1, 32, 0, st>>>(cnt, B, indptr);
  LR_LAUNCH_CHECK();
  sparsify_write_kernel<<<unsigned(B), SP_THREADS, 0, st>>>(reps, V, quant, thr, indptr, tok, impact, cap);
  LR_LAUNCH_CHECK();
  // nnz check (one small D2H): the caller sized `cap`; report overflow instead of silently truncating
  int32_t nnz = 0;
  LR_CUDA(cudaMemcpyAsync(&nnz, indptr + B, 4, cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaStreamSynchronize(st));
  if (int64_t(nnz) > cap) {
    set_error("sparsify: nnz %d exceeds capacity %lld", nnz, (long long)cap);
    return LR_EWORKSPACE;
  }
  return LR_OK;
}
