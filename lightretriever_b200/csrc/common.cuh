// common.cuh — error plumbing, key encoding and sm_100a PTX wrappers shared by the kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <limits.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/lr_b200.h"

namespace lr {

// ---------------------------------------------------------------- errors
void set_error(const char* fmt, ...);
#define LR_CHECK_ARG(cond, ...)                         \
  do {                                                  \
    if (!(cond)) {                                      \
      lr::set_error(__VA_ARGS__);                       \
      return LR_EINVAL;                                 \
    }                                                   \
  } while (0)
#define LR_CUDA(call)                                                              \
  do {                                                                             \
    cudaError_t _e = (call);                                                       \
    if (_e != cudaSuccess) {                                                       \
      lr::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return LR_ECUDA;                                                             \
    }                                                                              \
  } while (0)
#define LR_LAUNCH_CHECK()                                                          \
  do {                                                                             \
    cudaError_t _e = cudaGetLastError();                                           \
    if (_e != cudaSuccess) {                                                       \
      lr::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return LR_ECUDA;                                                             \
    }                                                                              \
    lr::count_launch();                                                            \
  } while (0)

void count_launch();  // one per kernel this library launched (lr_kernel_launches); defined in api.cu

int sm_count();  // cached per device

// optional CUDA events recorded around the dominant kernel of a call (lr_set_profile_events)
struct ProfileEvents {
  cudaEvent_t begin = nullptr, end = nullptr;
};
ProfileEvents& profile_events();  // thread-local, defined in api.cu

// Raises a kernel's dynamic shared-memory limit to at least `bytes`, once per (device, kernel).  The attribute belongs to
// the function, not to a stream: setting it per launch with that launch's own size races between host threads (one
// thread can lower it between another thread's set and launch).  Grow-only under a mutex; callers pass the most the
// kernel ever needs.  Defined in api.cu.
int ensure_dyn_smem(const void* func, int bytes);

// Tuning knobs (LR_* environment variables; the names and defaults are in knobs(), api.cu).  Production sets none of them.
// They are read once per thread and again after lr_reload_env(), which bumps env_epoch() so that the plan caches keyed
// on them are rebuilt too — tests flip knobs inside one process.
constexpr int KNOB_UNSET = INT_MIN;  // the variable is unset or empty: the planner derives the value from the shape
struct Knobs {
  // K2
  int flatip_prefix_docs;    // warm-start prefix in documents: 0 = single phase, < 0 = planner
  int flatip_cluster;        // 0 = planner, 1 = single CTA, 2 = cluster of 2 with multicast B, 3 = cta_group::2 pair
  int flatip_refresh;        // threshold-refresh passes: 0 / 1 = off / on for any prefix, < 0 = planner
  // K3
  int head_tiles_per_split;  // packed tokens: 256-token tiles per split (KNOB_UNSET = planner)
  int head_docs_per_unit;    // padded tokens: documents per split (KNOB_UNSET = planner)
  int head_sched;            // 0 = round robin only
  int head_team_band;        // row groups per band of the team schedule, 0 = no teams (KNOB_UNSET = planner)
  int head_team_window;      // tiles a team member may run ahead
  int head_cluster;          // as flatip_cluster
  // K4
  int sparse_kernel;         // 0 = by regime, 1 = flat kernel only, 3 = row kernel only
  bool sparse_acc32;         // int32 accumulators only (no 16-bit pass)
  bool sparse_debug;         // print the regime words and the overflow flag of every call (synchronises)
};
const Knobs& knobs();
unsigned env_epoch();

// ---------------------------------------------------------------- candidate keys
// A candidate is one u64: high word = order-preserving image of the score, low word =
// 0xFFFFFFFF - id, so that an unsigned descending sort yields (score desc, id asc).
__host__ __device__ __forceinline__ uint32_t f32_to_key(float f) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(f + 0.0f);  // -0 -> +0
#else
  float g = f + 0.0f;
  uint32_t u;
  memcpy(&u, &g, 4);
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float key_to_f32(uint32_t k) {
  uint32_t u = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}
__host__ __device__ __forceinline__ uint64_t make_key(uint32_t score_key, uint32_t id) {
  return (uint64_t(score_key) << 32) | uint64_t(0xFFFFFFFFu - id);
}
__host__ __device__ __forceinline__ uint32_t key_id(uint64_t k) { return 0xFFFFFFFFu - uint32_t(k); }
__host__ __device__ __forceinline__ uint32_t key_hi(uint64_t k) { return uint32_t(k >> 32); }
constexpr uint32_t KEY_NEG_INF = 0x007FFFFFu;  // f32_to_key(-inf)

// ---------------------------------------------------------------- document filters (lr_*_filtered, include/lr_b200.h)
// Bitmaps of u32 words indexed by GLOBAL document id (local row + id_offset): document i is allowed when bit i & 31 of
// word i >> 5 is set.  `live` (deletions) and the query's row of `allow` are ANDed; the kernels apply the filter before a
// document can enter a candidate list, so every threshold derived from a list is the k-th best of allowed documents.
struct DocFilter {
  const uint32_t* live;      // [ld_words] or null
  const uint32_t* allow;     // [n_filters][ld_words] or null
  const int32_t* q_filter;   // [Q] row of `allow` per query (-1 = unrestricted), or null = row 0 for every query
  int64_t ld_words;
  int64_t id_offset;         // global id of local row 0
  int n_filters;
  int on;                    // live || allow
};
constexpr int FILTER_ALL = -1;   // query filter row: no `allow` row applies
constexpr int FILTER_NONE = -2;  // query filter row: a q_filter outside [0, n_filters) allows nothing (fail closed)

// Validates the filter arguments of an N-row shard at id_offset and fills `f` (f.on == 0 when both bitmaps are null).
inline int make_doc_filter(const uint32_t* live, const uint32_t* allow, int64_t ld_words, int n_filters,
                           const int32_t* q_filter, int64_t id_offset, int64_t N, DocFilter& f) {
  f = DocFilter{live, allow, q_filter, ld_words, id_offset, n_filters, (live || allow) ? 1 : 0};
  LR_CHECK_ARG(!q_filter || allow, "filter: q_filter given without allow");
  LR_CHECK_ARG(!allow || n_filters >= 1, "filter: n_filters (%d) must be >= 1 with allow", n_filters);
  if (f.on)
    LR_CHECK_ARG(ld_words >= (id_offset + N + 31) / 32,
                 "filter: ld_words (%lld) must be >= ceil((id_offset + N) / 32) = %lld", (long long)ld_words,
                 (long long)((id_offset + N + 31) / 32));
  return LR_OK;
}

#ifdef __CUDACC__
// row of `allow` query q uses, FILTER_ALL or FILTER_NONE (32 bits: the K2 epilogue holds it in a register per unit)
__device__ __forceinline__ int filter_row(const DocFilter& f, int64_t q) {
  if (!f.allow) return FILTER_ALL;
  const int r = f.q_filter ? f.q_filter[q] : 0;
  if (r == -1) return FILTER_ALL;
  if (r < 0 || r >= f.n_filters) return FILTER_NONE;
  return r;
}
// bits [id, id + 32) of a bitmap (bit j = document id + j); words past ld_words read as 0.  An id that is not a multiple
// of 32 spans two words: funnel shift.
__device__ __forceinline__ uint32_t bitmap_bits32(const uint32_t* w, int64_t ld_words, int64_t id) {
  const int64_t wi = id >> 5;
  const int sh = int(id & 31);
  const uint32_t lo = wi < ld_words ? w[wi] : 0u;
  if (sh == 0) return lo;
  const uint32_t hi = wi + 1 < ld_words ? w[wi + 1] : 0u;
  return __funnelshift_r(lo, hi, sh);
}
// allowed-mask of the 32 documents at local rows [col, col + 32)
__device__ __forceinline__ uint32_t filter_mask32(const DocFilter& f, int row, int64_t col) {
  if (row == FILTER_NONE) return 0u;
  const int64_t id = f.id_offset + col;
  uint32_t m = f.live ? bitmap_bits32(f.live, f.ld_words, id) : 0xFFFFFFFFu;
  if (row >= 0) m &= bitmap_bits32(f.allow + int64_t(row) * f.ld_words, f.ld_words, id);
  return m;
}
// whether the document at local row `col` is allowed
__device__ __forceinline__ bool filter_allows(const DocFilter& f, int row, int64_t col) {
  if (row == FILTER_NONE) return false;
  const int64_t id = f.id_offset + col;
  const uint32_t bit = 1u << (id & 31);
  if (f.live && !(f.live[id >> 5] & bit)) return false;
  return row < 0 || (f.allow[int64_t(row) * f.ld_words + (id >> 5)] & bit) != 0;
}
#endif  // __CUDACC__

#ifdef __CUDACC__
// ---------------------------------------------------------------- cache-hinted global access
__device__ __forceinline__ uint64_t ld_cg_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_cg_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.global.cg.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add_u32(uint32_t* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 ld_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// ---------------------------------------------------------------- shared / mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// The suspend-time hint lets the hardware park the warp until the phase completes (or the hint expires) instead of
// returning at once: the single-lane producer / MMA warps share their schedulers with epilogue warps, and a tight
// try_wait spin takes issue slots from them (ncu, MRL shapes: 17 % of all issued instructions were this loop).
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(1000000u)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU.
#ifndef LR_MBAR_TIMEOUT_CYCLES
#define LR_MBAR_TIMEOUT_CYCLES (20ll * 1000 * 1000 * 1000)
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3FFu) == 0 && clock64() - t0 > LR_MBAR_TIMEOUT_CYCLES) {
      printf("lr_b200: mbarrier timeout block %d thread %d bar %u parity %u\n", blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
// multicast variant: the box lands at the same CTA-relative offset in every CTA of `mask`, and each destination's
// mbarrier (same offset) receives the complete_tx
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar,
                                               uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc_hint(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar,
                                                    uint16_t mask, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5, %6;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "h"(mask), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// ---- 2-SM (cta_group::2) forms: the CTA pair of a cluster cooperates on one M=256 MMA
// shared::cluster address of `addr` (a shared::cta address of this CTA) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// TMA load into THIS CTA's shared memory whose completion bytes are counted on an mbarrier of the pair's leader CTA
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t leader_bar,
                                                uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
// Arrive on an mbarrier of another CTA of the cluster.  Default semantics (.release at CTA scope), as CUTLASS's
// ClusterBarrier::arrive: the barriers signalled this way order TMEM reads against later MMAs through the tcgen05
// fences around them, not through generic-proxy memory, and a cluster-scope release costs an L1 invalidation per arrive
// (ncu, MRL shapes: 9 % of all stall samples sat on this one instruction).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// createpolicy constant (same encoding CUTLASS uses for TMA::CacheHintSm90::EVICT_NORMAL)
constexpr uint64_t L2_EVICT_NORMAL = 0x1000000000000000ull;

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem] . B[smem]^T, bf16 x bf16 -> f32, issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all previously issued tcgen05.mma of this thread completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 consecutive f32 columns: thread i of the warp receives lane (taddr.lane + i)
// same, arriving on the barrier at this offset in every CTA of `mask` (a slot shared through multicast is free only
// when all CTAs of the cluster have read it)
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask) : "memory");
}
// cta_group::2 variants (issued by the leader CTA's MMA thread / both CTAs' allocator warps)
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2sm_mc(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (rows of 128 bytes, 8-row groups of 1024 bytes).
// Bit layout: cute::UMMA::SmemDescriptor (start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48),
// layout_type [61,64) with SWIZZLE_128B = 2).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  return uint64_t((smem_addr >> 4) & 0x3FFFu) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
// kind::f16 instruction descriptor: f32 accumulate, bf16 A/B, both K-major (cute::UMMA::InstrDescriptor).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}

// One warp scans a 256-bin histogram from the top bin down and finds the bin holding the `remaining`-th
// largest element.  Returns (bin, rank inside the bin, whether the bin is taken whole) in every lane.
__device__ __forceinline__ void warp_find_bin_desc(const uint32_t* hist, uint32_t remaining, uint32_t& bin,
                                                   uint32_t& rem2, bool& take_all) {
  const uint32_t full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const int base = 8 * (31 - lane);  // lane 0 owns the highest bins
  uint32_t c[8], sum = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    c[i] = hist[base + 7 - i];
    sum += c[i];
  }
  uint32_t incl = sum;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const uint32_t t = __shfl_up_sync(full, incl, off);
    if (lane >= off) incl += t;
  }
  const uint32_t excl = incl - sum;
  const bool hit = (excl < remaining) && (remaining <= incl);
  const uint32_t hm = __ballot_sync(full, hit);
  const int src = hm ? (__ffs(hm) - 1) : 31;
  uint32_t b = 0, r = 1, ta = 0;
  if (lane == src) {
    uint32_t acc = excl;
    bool done = false;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (!done && acc + c[i] >= remaining) {
        b = uint32_t(base + 7 - i);
        r = remaining - acc;
        ta = (c[i] == r) ? 1u : 0u;
        done = true;
      }
      if (!done) acc += c[i];
    }
  }
  bin = __shfl_sync(full, b, src);
  rem2 = __shfl_sync(full, r, src);
  take_all = __shfl_sync(full, ta, src) != 0;
}

__device__ __forceinline__ uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}
#endif  // __CUDACC__

}  // namespace lr
