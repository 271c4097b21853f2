// embbag.cu — K1: EmbeddingBag (mean, padding_idx) + MRL truncate + L2 normalise, fused; K1b last-token head.
//
// Replaces  self.emb_bag.forward(input, offsets)      reference finetune/modeling_hybrid.py:474
//           emb_reps[..., :dense_shrink_dim]           finetune/modeling_hybrid.py:487-488
//           F.normalize(emb_reps, p=2, dim=-1)         finetune/modeling_hybrid.py:489-490
// and       pooling(..., 'lasttoken') + shrink + normalize   finetune/dense_pooling.py:48-55,
//                                                             finetune/modeling_hybrid.py:266-278
//
// HBM-bound gather: one CTA per bag; every thread owns 16-byte column chunks (8 bf16 / 4 f32) and walks the
// bag's rows four at a time so that >= 4 independent 16-byte loads per thread are in flight.  Only the first
// out_dim columns are read (MRL prefix).  Accumulation is fp32 in token order; the mean, the squared norm and
// the scaling happen in registers / shared memory, so the row is written exactly once.
#include "common.cuh"

namespace lr {

constexpr int EB_THREADS = 128;
constexpr int EB_MAX_TOKENS_SMEM = 1024;  // ids cached in shared memory; longer bags re-read from global
// widest out_dim the entry points accept.  A block kernel's float row[out_dim] plus its static shared memory (the 8 KiB id
// cache of embbag_kernel, 16 B in lasttoken_gather_kernel) can exceed the 48 KiB a launch gets without opting in, so
// both entry points raise each kernel's limit to this width once.
constexpr int EB_MAX_OUT_DIM = 12288;

template <typename T>
struct Vec16;
template <>
struct Vec16<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void add(const uint4& r, float (&acc)[8]) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      acc[2 * i] += __uint_as_float(w[i] << 16);
      acc[2 * i + 1] += __uint_as_float(w[i] & 0xFFFF0000u);
    }
  }
  static __device__ __forceinline__ void load_add(const __nv_bfloat16* p, float (&acc)[8]) { add(ld_nc_v4(p), acc); }
};
template <>
struct Vec16<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void add(const uint4& r, float (&acc)[4]) {
    acc[0] += __uint_as_float(r.x);
    acc[1] += __uint_as_float(r.y);
    acc[2] += __uint_as_float(r.z);
    acc[3] += __uint_as_float(r.w);
  }
  static __device__ __forceinline__ void load_add(const float* p, float (&acc)[4]) { add(ld_nc_v4(p), acc); }
};

template <typename TO>
__device__ __forceinline__ void store_out(TO* p, float v);
template <>
__device__ __forceinline__ void store_out<float>(float* p, float v) { *p = v; }
template <>
__device__ __forceinline__ void store_out<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, off);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
  for (int w = 0; w < EB_THREADS / 32; ++w) t += red[w];
  __syncthreads();
  return t;
}

// table [V, d]; one CTA per bag; dynamic smem: float row[out_dim]
template <typename TT, typename TO>
__global__ void __launch_bounds__(EB_THREADS)
embbag_kernel(const int64_t* __restrict__ ids, const int64_t* __restrict__ offsets, int64_t n_ids, int64_t n_bags,
              const TT* __restrict__ table, int64_t V, int64_t d, int64_t padding_idx, int out_dim, int normalize,
              TO* __restrict__ out, int32_t* err_flag) {
  extern __shared__ float row[];
  __shared__ int64_t s_ids[EB_MAX_TOKENS_SMEM];
  __shared__ float red[EB_THREADS / 32];
  __shared__ int s_cnt, s_bad;
  constexpr int VN = Vec16<TT>::N;
  const int64_t bag = blockIdx.x;
  const int64_t beg = offsets[bag];
  const int64_t end = (bag + 1 < n_bags) ? offsets[bag + 1] : n_ids;
  const int64_t len = end > beg ? end - beg : 0;
  const int tid = threadIdx.x;
  if (tid == 0) {
    s_cnt = 0;
    s_bad = 0;
  }
  __syncthreads();
  // stage ids, drop padding, validate
  const bool cached = len <= EB_MAX_TOKENS_SMEM;
  int local_cnt = 0, local_bad = 0;
  for (int64_t i = tid; i < len; i += EB_THREADS) {
    int64_t id = ids[beg + i];
    if (id != padding_idx) {
      ++local_cnt;
      if (id < 0 || id >= V) {
        local_bad = 1;
        id = -1;
      }
    } else {
      id = -1;  // skipped
    }
    if (cached) s_ids[i] = id;
  }
  if (local_cnt) atomicAdd(&s_cnt, local_cnt);
  if (local_bad) atomicOr(&s_bad, 1);
  __syncthreads();
  const int cnt = s_cnt;
  const bool bad = s_bad != 0;

  const int nchunks = out_dim / VN;
  float sumsq = 0.f;
  for (int c = tid; c < nchunks; c += EB_THREADS) {
    float acc[VN];
#pragma unroll
    for (int i = 0; i < VN; ++i) acc[i] = 0.f;
    const TT* col = table + int64_t(c) * VN;
    int64_t i = 0;
    if (cached) {
      // eight, then four independent 16-byte loads in flight (skipped ids read row 0 and are discarded); token order is
      // preserved: the adds are issued in index order
      for (; i + 8 <= len; i += 8) {
        int64_t t[8];
        uint4 r[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) t[u] = s_ids[i + u];
#pragma unroll
        for (int u = 0; u < 8; ++u) r[u] = ld_nc_v4(col + (t[u] >= 0 ? t[u] : 0) * d);
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (t[u] >= 0) Vec16<TT>::add(r[u], acc);
      }
      for (; i + 4 <= len; i += 4) {
        const int64_t a = s_ids[i], b = s_ids[i + 1], e = s_ids[i + 2], f = s_ids[i + 3];
        const uint4 ra = ld_nc_v4(col + (a >= 0 ? a : 0) * d);
        const uint4 rb = ld_nc_v4(col + (b >= 0 ? b : 0) * d);
        const uint4 re = ld_nc_v4(col + (e >= 0 ? e : 0) * d);
        const uint4 rf = ld_nc_v4(col + (f >= 0 ? f : 0) * d);
        if (a >= 0) Vec16<TT>::add(ra, acc);
        if (b >= 0) Vec16<TT>::add(rb, acc);
        if (e >= 0) Vec16<TT>::add(re, acc);
        if (f >= 0) Vec16<TT>::add(rf, acc);
      }
      for (; i < len; ++i) {
        const int64_t a = s_ids[i];
        if (a >= 0) Vec16<TT>::load_add(col + a * d, acc);
      }
    } else {
      for (; i < len; ++i) {
        const int64_t a = ids[beg + i];
        if (a != padding_idx && a >= 0 && a < V) Vec16<TT>::load_add(col + a * d, acc);
      }
    }
#pragma unroll
    for (int j = 0; j < VN; ++j) {
      // torch divides the fp32 sum by the count (aten EmbeddingBag mean)
      const float m = cnt > 0 ? acc[j] / float(cnt) : 0.0f;
      row[c * VN + j] = m;
      sumsq += m * m;
    }
  }
  float scale = 1.0f;
  if (normalize) {
    const float tot = block_sum(sumsq, red);
    scale = 1.0f / fmaxf(sqrtf(tot), 1e-12f);
  } else {
    __syncthreads();
  }
  TO* o = out + bag * int64_t(out_dim);
  for (int c = tid; c < nchunks; c += EB_THREADS) {
#pragma unroll
    for (int j = 0; j < VN; ++j) {
      float v = row[c * VN + j];
      // F.normalize divides by max(norm, eps)
      v = normalize ? v * scale : v;
      if (bad) v = __int_as_float(0x7FC00000);
      store_out<TO>(o + c * VN + j, v);
    }
  }
  if (bad && tid == 0 && err_flag) atomicOr(err_flag, 1);
}

// Narrow outputs (MRL prefixes of <= 32 16-byte chunks: 256 bf16 / 128 f32 columns): one WARP per bag, four bags per
// CTA, no shared memory and no block barrier — a CTA per bag would leave 3/4 of its threads idle and spend its life in
// the id-staging and reduction barriers.  Lane c owns chunk c; the ids of 32 tokens are staged one per lane and
// broadcast by shuffle; eight row loads per lane are in flight; adds stay in token order.
template <typename TT, typename TO>
__global__ void __launch_bounds__(EB_THREADS)
embbag_warp_kernel(const int64_t* __restrict__ ids, const int64_t* __restrict__ offsets, int64_t n_ids, int64_t n_bags,
                   const TT* __restrict__ table, int64_t V, int64_t d, int64_t padding_idx, int out_dim, int normalize,
                   TO* __restrict__ out, int32_t* err_flag) {
  constexpr int VN = Vec16<TT>::N;
  const uint32_t full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const int64_t bag = int64_t(blockIdx.x) * (EB_THREADS / 32) + (threadIdx.x >> 5);
  if (bag >= n_bags) return;
  const int64_t beg = offsets[bag];
  const int64_t end = (bag + 1 < n_bags) ? offsets[bag + 1] : n_ids;
  const int64_t len = end > beg ? end - beg : 0;
  const int nchunks = out_dim / VN;  // <= 32
  const bool active = lane < nchunks;
  const TT* col = table + int64_t(active ? lane : 0) * VN;
  float acc[VN];
#pragma unroll
  for (int i = 0; i < VN; ++i) acc[i] = 0.f;
  int cnt = 0;
  bool bad = false;
  for (int64_t base = 0; base < len; base += 32) {
    int64_t id = -1;  // -1: skipped (padding, invalid, past the end)
    if (base + lane < len) {
      id = ids[beg + base + lane];
      if (id == padding_idx) {
        id = -1;
      } else if (id < 0 || id >= V) {
        bad = true;
        id = -2;  // counted like torch counts it, never read
      }
    }
    cnt += __popc(__ballot_sync(full, id != -1));
    const int nb = int(len - base < 32 ? len - base : 32);
    for (int u0 = 0; u0 < nb; u0 += 8) {
      int64_t t[8];
      uint4 r[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) t[u] = __shfl_sync(full, id, (u0 + u) & 31);
#pragma unroll
      for (int u = 0; u < 8; ++u) r[u] = ld_nc_v4(col + (t[u] >= 0 ? t[u] : 0) * d);
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (u0 + u < nb && t[u] >= 0) Vec16<TT>::add(r[u], acc);
    }
  }
  bad = __any_sync(full, bad);
  float sumsq = 0.f;
#pragma unroll
  for (int j = 0; j < VN; ++j) {
    acc[j] = (cnt > 0 && active) ? acc[j] / float(cnt) : 0.0f;  // torch divides the fp32 sum by the count
    sumsq += acc[j] * acc[j];
  }
  float scale = 1.0f;
  if (normalize) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sumsq += __shfl_xor_sync(full, sumsq, off);
    scale = 1.0f / fmaxf(sqrtf(sumsq), 1e-12f);  // F.normalize divides by max(norm, eps)
  }
  if (active) {
    TO* o = out + bag * int64_t(out_dim) + lane * VN;
#pragma unroll
    for (int j = 0; j < VN; ++j) store_out<TO>(o + j, bad ? __int_as_float(0x7FC00000) : acc[j] * scale);
  }
  if (bad && lane == 0 && err_flag) atomicOr(err_flag, 1);
}

// ---- K1b: last-token index (dense_pooling.py:48-55)
__global__ void lasttoken_index_kernel(const int64_t* __restrict__ mask, int64_t B, int64_t S, int32_t* scratch) {
  // scratch[0..B) = sum(mask[b]) - 1 ; scratch[B] = number of rows whose last column is valid
  const int64_t b = blockIdx.x;
  long long s = 0;
  for (int64_t i = threadIdx.x; i < S; i += blockDim.x) s += mask[b * S + i];
  __shared__ long long red[32];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long t = 0;
    for (int w = 0; w < int(blockDim.x >> 5); ++w) t += red[w];
    scratch[b] = int32_t(t - 1);
    // torch: attention_mask[:, -1].sum() == B  (mask values are 0/1)
    atomicAdd(scratch + B, int32_t(mask[b * S + S - 1]));
  }
}

template <typename TT, typename TO>
__global__ void __launch_bounds__(EB_THREADS)
lasttoken_gather_kernel(const TT* __restrict__ hidden, int64_t B, int64_t S, int64_t d, const int32_t* scratch,
                        int out_dim, int normalize, TO* __restrict__ out) {
  extern __shared__ float row[];
  __shared__ float red[EB_THREADS / 32];
  constexpr int VN = Vec16<TT>::N;
  const int64_t b = blockIdx.x;
  const bool left_padding = scratch[B] == int32_t(B);
  int64_t idx = left_padding ? S - 1 : int64_t(scratch[b]);
  if (idx < 0) idx += S;  // torch negative index wraps
  const TT* src = hidden + (b * S + idx) * d;
  const int nchunks = out_dim / VN;
  float sumsq = 0.f;
  for (int c = threadIdx.x; c < nchunks; c += EB_THREADS) {
    float acc[VN];
#pragma unroll
    for (int i = 0; i < VN; ++i) acc[i] = 0.f;
    Vec16<TT>::load_add(src + int64_t(c) * VN, acc);
#pragma unroll
    for (int j = 0; j < VN; ++j) {
      row[c * VN + j] = acc[j];
      sumsq += acc[j] * acc[j];
    }
  }
  float scale = 1.0f;
  if (normalize) {
    const float tot = block_sum(sumsq, red);
    scale = 1.0f / fmaxf(sqrtf(tot), 1e-12f);
  } else {
    __syncthreads();
  }
  TO* o = out + b * int64_t(out_dim);
  for (int c = threadIdx.x; c < nchunks; c += EB_THREADS)
#pragma unroll
    for (int j = 0; j < VN; ++j) store_out<TO>(o + c * VN + j, normalize ? row[c * VN + j] * scale : row[c * VN + j]);
}

}  // namespace lr

using namespace lr;

extern "C" int lr_embbag_encode(const int64_t* ids, const int64_t* offsets, int64_t n_ids, int64_t n_bags,
                                const void* table, int table_dtype, int64_t V, int64_t d, int64_t padding_idx,
                                int64_t out_dim, int normalize, void* out, int out_dtype, int32_t* err_flag,
                                void* stream) {
  LR_CHECK_ARG(n_bags >= 0 && n_ids >= 0, "embbag: negative sizes");
  if (n_bags == 0) return LR_OK;
  LR_CHECK_ARG(offsets && table && out, "embbag: null pointer");
  LR_CHECK_ARG(ids || n_ids == 0, "embbag: null ids");
  LR_CHECK_ARG(table_dtype == LR_BF16 || table_dtype == LR_F32, "embbag: table_dtype must be LR_BF16 or LR_F32");
  LR_CHECK_ARG(out_dtype == LR_BF16 || out_dtype == LR_F32, "embbag: out_dtype must be LR_BF16 or LR_F32");
  const int esz = table_dtype == LR_BF16 ? 2 : 4;
  LR_CHECK_ARG(V >= 1 && d >= 1 && (d * esz) % 16 == 0, "embbag: table rows must be a multiple of 16 bytes (d=%lld)",
               (long long)d);
  LR_CHECK_ARG((uintptr_t(table) & 15) == 0, "embbag: table must be 16-byte aligned");
  LR_CHECK_ARG(out_dim >= 8 && out_dim <= d && out_dim % 8 == 0, "embbag: out_dim (%lld) must be a multiple of 8 in [8, d]",
               (long long)out_dim);
  LR_CHECK_ARG(out_dim <= EB_MAX_OUT_DIM, "embbag: out_dim (%lld) too large", (long long)out_dim);
  LR_CHECK_ARG(n_bags < (int64_t(1) << 31), "embbag: too many bags");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t smem = size_t(out_dim) * 4;
  const dim3 grid{unsigned(n_bags)};
#define LR_EB_LAUNCH(TT, TO)                                                                                     \
  do {                                                                                                           \
    const int rc = ensure_dyn_smem(reinterpret_cast<const void*>(embbag_kernel<TT, TO>), EB_MAX_OUT_DIM * 4);    \
    if (rc) return rc;                                                                                           \
    embbag_kernel<TT, TO><<<grid, EB_THREADS, smem, st>>>(ids, offsets, n_ids, n_bags, static_cast<const TT*>(table), \
                                                          V, d, padding_idx, int(out_dim), normalize,            \
                                                          static_cast<TO*>(out), err_flag);                      \
  } while (0)
  const int vn = table_dtype == LR_BF16 ? 8 : 4;
  const bool narrow = out_dim / vn <= 32;  // one warp per bag
  const dim3 wgrid{unsigned((n_bags + EB_THREADS / 32 - 1) / (EB_THREADS / 32))};
#define LR_EBW_LAUNCH(TT, TO)                                                                                     \
  embbag_warp_kernel<TT, TO><<<wgrid, EB_THREADS, 0, st>>>(ids, offsets, n_ids, n_bags, static_cast<const TT*>(table), \
                                                           V, d, padding_idx, int(out_dim), normalize,          \
                                                           static_cast<TO*>(out), err_flag)
  if (narrow) {
    if (table_dtype == LR_BF16 && out_dtype == LR_BF16) LR_EBW_LAUNCH(__nv_bfloat16, __nv_bfloat16);
    else if (table_dtype == LR_BF16) LR_EBW_LAUNCH(__nv_bfloat16, float);
    else if (out_dtype == LR_BF16) LR_EBW_LAUNCH(float, __nv_bfloat16);
    else LR_EBW_LAUNCH(float, float);
  } else if (table_dtype == LR_BF16 && out_dtype == LR_BF16) LR_EB_LAUNCH(__nv_bfloat16, __nv_bfloat16);
  else if (table_dtype == LR_BF16) LR_EB_LAUNCH(__nv_bfloat16, float);
  else if (out_dtype == LR_BF16) LR_EB_LAUNCH(float, __nv_bfloat16);
  else LR_EB_LAUNCH(float, float);
#undef LR_EB_LAUNCH
#undef LR_EBW_LAUNCH
  LR_LAUNCH_CHECK();
  return LR_OK;
}

extern "C" int lr_lasttoken_head(const void* hidden, int hidden_dtype, const int64_t* mask, int64_t B, int64_t S,
                                 int64_t d, int64_t out_dim, int normalize, void* out, int out_dtype,
                                 int32_t* scratch, void* stream) {
  LR_CHECK_ARG(B >= 0, "lasttoken: negative batch");
  if (B == 0) return LR_OK;
  LR_CHECK_ARG(hidden && mask && out && scratch, "lasttoken: null pointer");
  LR_CHECK_ARG(hidden_dtype == LR_BF16 || hidden_dtype == LR_F32, "lasttoken: bad hidden dtype");
  LR_CHECK_ARG(out_dtype == LR_BF16 || out_dtype == LR_F32, "lasttoken: bad out dtype");
  const int esz = hidden_dtype == LR_BF16 ? 2 : 4;
  LR_CHECK_ARG(S >= 1 && d >= 1 && (d * esz) % 16 == 0 && (uintptr_t(hidden) & 15) == 0,
               "lasttoken: hidden rows must be 16-byte aligned multiples of 16 bytes");
  LR_CHECK_ARG(out_dim >= 8 && out_dim <= d && out_dim % 8 == 0 && out_dim <= EB_MAX_OUT_DIM,
               "lasttoken: out_dim (%lld) must be a multiple of 8 in [8, d]", (long long)out_dim);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LR_CUDA(cudaMemsetAsync(scratch + B, 0, 4, st));
  lasttoken_index_kernel<<<unsigned(B), 128, 0, st>>>(mask, B, S, scratch);
  LR_LAUNCH_CHECK();
  const size_t smem = size_t(out_dim) * 4;
#define LR_LT_LAUNCH(TT, TO)                                                                                       \
  do {                                                                                                             \
    const int rc = ensure_dyn_smem(reinterpret_cast<const void*>(lasttoken_gather_kernel<TT, TO>), EB_MAX_OUT_DIM * 4); \
    if (rc) return rc;                                                                                             \
    lasttoken_gather_kernel<TT, TO><<<unsigned(B), EB_THREADS, smem, st>>>(static_cast<const TT*>(hidden), B, S, d, \
                                                                           scratch, int(out_dim), normalize,        \
                                                                           static_cast<TO*>(out));                  \
  } while (0)
  if (hidden_dtype == LR_BF16 && out_dtype == LR_BF16) LR_LT_LAUNCH(__nv_bfloat16, __nv_bfloat16);
  else if (hidden_dtype == LR_BF16) LR_LT_LAUNCH(__nv_bfloat16, float);
  else if (out_dtype == LR_BF16) LR_LT_LAUNCH(float, __nv_bfloat16);
  else LR_LT_LAUNCH(float, float);
#undef LR_LT_LAUNCH
  LR_LAUNCH_CHECK();
  return LR_OK;
}
