// groupby.cu — the session-based path (sm_100a): Groupby, ListSlice and the row ordering behind
// Dataset.shuffle_by_keys.  The reference gets these from cuDF (sort_values + groupby.agg +
// list.get, nvtabular/ops/groupby.py:114-150,213-240,290-319) and from two numba kernels
// (_calculate_row_sizes / _slice_rows, nvtabular/ops/list_slice.py:180-228).
//
//   nvtb_sort_rows          stable lexicographic row order: LSD over the key columns, one
//                           radix.cuh sort of (digit << 32 | position) words per 32-bit key word,
//                           passes trimmed to each key's value range, 1-bit null-flag passes
//   nvtb_segments           group boundaries of the sorted keys (flag + scan + scatter)
//   nvtb_gather_rows        typed gather of a column (+ validity) through the permutation
//   nvtb_segment_agg        count/sum/mean/min/max/std/var/first/last of every group: groups of
//                           <= kShortMax rows take one thread, longer groups are cut into chunks
//                           of kChunk rows, each reduced by a CTA and merged with atomics
//   nvtb_segment_sorted_agg median / nunique over groups whose values are sorted (nulls last)
//   nvtb_list_slice_*       per-row slice sizes + scan, then a load-balanced element copy
#include "common.cuh"
#include "radix.cuh"

namespace nvtb {
namespace {

constexpr int kGbThreads = 256;
constexpr int kScanItems = 16;
constexpr int kScanTile = kGbThreads * kScanItems;     // rows per scan tile
constexpr int kShortMax = 32;                          // longest group one thread reduces alone
constexpr int kChunkItems = 8;
constexpr int kChunk = kGbThreads * kChunkItems;       // rows per CTA on the long-group path
constexpr int kMaxKeys = 8;

inline int gb_grid(int64_t work) {
  int64_t b = (work + kGbThreads - 1) / kGbThreads;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// ------------------------------------------------------------------------------------ images
// order-preserving unsigned image of a value (sorting and group equality: -0.0 == +0.0)
__device__ __forceinline__ uint64_t sort_image(const void* data, int dt, int64_t i) {
  switch (dt) {
    case NVTB_I32: return (uint64_t)((uint32_t)((const int32_t*)data)[i] ^ 0x80000000u);
    case NVTB_I64: return (uint64_t)((const int64_t*)data)[i] ^ 0x8000000000000000ull;
    case NVTB_F32: {
      const float f = ((const float*)data)[i];
      const uint32_t u = f == 0.0f ? 0u : __float_as_uint(f);
      return (uint64_t)((u & 0x80000000u) ? ~u : (u | 0x80000000u));
    }
    case NVTB_F64: {
      const double f = ((const double*)data)[i];
      const uint64_t u = f == 0.0 ? 0ull : (uint64_t)__double_as_longlong(f);
      return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
    }
    default: return (uint64_t)((const uint8_t*)data)[i];
  }
}

// exact typed image for min / max (decoded back with from_image)
template <typename T> __device__ __forceinline__ uint64_t to_image(T x);
template <> __device__ __forceinline__ uint64_t to_image<int32_t>(int32_t x) { return (uint64_t)((uint32_t)x ^ 0x80000000u); }
template <> __device__ __forceinline__ uint64_t to_image<int64_t>(int64_t x) { return (uint64_t)x ^ 0x8000000000000000ull; }
template <> __device__ __forceinline__ uint64_t to_image<uint8_t>(uint8_t x) { return (uint64_t)x; }
template <> __device__ __forceinline__ uint64_t to_image<float>(float x) {
  const uint32_t u = __float_as_uint(x);
  return (uint64_t)((u & 0x80000000u) ? ~u : (u | 0x80000000u));
}
template <> __device__ __forceinline__ uint64_t to_image<double>(double x) {
  const uint64_t u = (uint64_t)__double_as_longlong(x);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
template <typename T> __device__ __forceinline__ T from_image(uint64_t m);
template <> __device__ __forceinline__ int32_t from_image<int32_t>(uint64_t m) { return (int32_t)((uint32_t)m ^ 0x80000000u); }
template <> __device__ __forceinline__ int64_t from_image<int64_t>(uint64_t m) { return (int64_t)(m ^ 0x8000000000000000ull); }
template <> __device__ __forceinline__ uint8_t from_image<uint8_t>(uint64_t m) { return (uint8_t)m; }
template <> __device__ __forceinline__ float from_image<float>(uint64_t m) {
  const uint32_t u = (uint32_t)m;
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}
template <> __device__ __forceinline__ double from_image<double>(uint64_t m) {
  return __longlong_as_double((long long)((m >> 63) ? (m & 0x7FFFFFFFFFFFFFFFull) : ~m));
}

// -------------------------------------------------------------------------- block reductions
__device__ __forceinline__ int64_t warp_sum(int64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
  return v;
}

// exclusive scan of one int64 per thread over the block; returns the block total to all threads
__device__ __forceinline__ int64_t block_excl_scan(int64_t v, int64_t* excl) {
  __shared__ int64_t ws[kGbThreads / 32 + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) ws[warp] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t run = 0;
    for (int w = 0; w < kGbThreads / 32; ++w) { const int64_t t = ws[w]; ws[w] = run; run += t; }
    ws[kGbThreads / 32] = run;
  }
  __syncthreads();
  *excl = ws[warp] + incl - v;
  const int64_t total = ws[kGbThreads / 32];
  __syncthreads();
  return total;
}

// ---------------------------------------------------------------------- device-wide scan
// Exclusive scan of v(i), i < n (n = *n_dev when n_dev != NULL, capped at n_max); every item
// is handed to sink(i, prefix, value).  Three kernels: tile sums, scan of the tile sums (one
// CTA; the grand total goes to *total), tile-local scans.
template <class V>
__global__ void __launch_bounds__(kGbThreads) scan_reduce_kernel(V v, const int64_t* n_dev, int64_t n_max,
                                                                 int64_t* tile_sums) {
  __shared__ int64_t ws[kGbThreads / 32];
  const int64_t n = n_dev ? (*n_dev < n_max ? *n_dev : n_max) : n_max;
  const int64_t base = (int64_t)blockIdx.x * kScanTile;
  int64_t s = 0;
#pragma unroll 4
  for (int j = 0; j < kScanItems; ++j) {
    const int64_t i = base + (int64_t)j * kGbThreads + threadIdx.x;
    if (i < n) s += v(i);
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t t = 0;
    for (int w = 0; w < kGbThreads / 32; ++w) t += ws[w];
    tile_sums[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(kGbThreads) scan_tiles_kernel(int64_t* tile_sums, int64_t T, int64_t* total) {
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t c0 = 0; c0 < T; c0 += kGbThreads) {
    const int64_t i = c0 + threadIdx.x;
    const int64_t v = i < T ? tile_sums[i] : 0;
    int64_t ex;
    const int64_t tot = block_excl_scan(v, &ex);
    if (i < T) tile_sums[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

template <class V, class S>
__global__ void __launch_bounds__(kGbThreads) scan_apply_kernel(V v, S sink, const int64_t* n_dev, int64_t n_max,
                                                                const int64_t* tile_sums) {
  const int64_t n = n_dev ? (*n_dev < n_max ? *n_dev : n_max) : n_max;
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  // v is evaluated twice (the second time from L1/L2) rather than kept: 16 int64 per thread spill
  int64_t local = 0;
  for (int j = 0; j < kScanItems; ++j) {
    const int64_t i = base + j;
    if (i < n) local += v(i);
  }
  int64_t ex;
  block_excl_scan(local, &ex);
  int64_t run = tile_sums[blockIdx.x] + ex;
  for (int j = 0; j < kScanItems; ++j) {
    const int64_t i = base + j;
    if (i < n) {
      const int64_t x = v(i);
      sink(i, run, x);
      run += x;
    }
  }
}

// scan scratch: tile sums + total
struct ScanScratch {
  int64_t* tiles;
  int64_t* total;
  int64_t T;
};
inline int64_t scan_tiles(int64_t n_max) { return (n_max + kScanTile - 1) / kScanTile; }

template <class V, class S>
int device_scan(V v, S sink, const int64_t* n_dev, int64_t n_max, const ScanScratch& sc, cudaStream_t st) {
  if (n_max <= 0) {
    NVTB_CUDA_OK(cudaMemsetAsync(sc.total, 0, sizeof(int64_t), st));
    return NVTB_OK;
  }
  scan_reduce_kernel<V><<<(unsigned)sc.T, kGbThreads, 0, st>>>(v, n_dev, n_max, sc.tiles);
  NVTB_LAUNCH_OK();
  scan_tiles_kernel<<<1, kGbThreads, 0, st>>>(sc.tiles, sc.T, sc.total);
  NVTB_LAUNCH_OK();
  scan_apply_kernel<V, S><<<(unsigned)sc.T, kGbThreads, 0, st>>>(v, sink, n_dev, n_max, sc.tiles);
  NVTB_LAUNCH_OK();
  return NVTB_OK;
}

int scan_alloc(ScanScratch* sc, int64_t n_max, cudaStream_t st) {
  sc->T = scan_tiles(n_max);
  void* p = nullptr;
  NVTB_CUDA_OK(cudaMallocAsync(&p, sizeof(int64_t) * (size_t)(sc->T + 2), st));
  sc->total = reinterpret_cast<int64_t*>(p);
  sc->tiles = sc->total + 1;
  return NVTB_OK;
}

// ------------------------------------------------------------------------------- row sort
__global__ void identity_kernel(uint64_t* e, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    e[i] = (uint64_t)i;
}

// min / max of the sort image over the valid rows (mins[k] starts at ~0, maxs[k] at 0)
__global__ void __launch_bounds__(kGbThreads) key_range_kernel(nvtb_col_t c, int64_t n, unsigned long long* mn,
                                                               unsigned long long* mx) {
  uint64_t lo = ~0ull, hi = 0ull;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (!valid1(c.validity, i)) continue;
    const uint64_t m = sort_image(c.data, c.dtype, i);
    lo = m < lo ? m : lo;
    hi = m > hi ? m : hi;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const uint64_t a = __shfl_down_sync(0xFFFFFFFFu, lo, o), b = __shfl_down_sync(0xFFFFFFFFu, hi, o);
    lo = a < lo ? a : lo;
    hi = b > hi ? b : hi;
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(mn, (unsigned long long)lo);
    atomicMax(mx, (unsigned long long)hi);
  }
}

// high word of every element := digit of the key at the element's row (position = low word)
__global__ void set_digit_kernel(uint64_t* e, int64_t n, nvtb_col_t c, uint64_t base, int desc, int shift) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t pos = (uint32_t)e[i];
    uint32_t d = 0;
    if (valid1(c.validity, pos)) {
      const uint64_t m = sort_image(c.data, c.dtype, pos);
      d = (uint32_t)((desc ? base - m : m - base) >> shift);
    }
    e[i] = ((uint64_t)d << 32) | pos;
  }
}

struct Masks {
  const uint8_t* v[kMaxKeys];
  int n;
};

__global__ void set_null_digit_kernel(uint64_t* e, int64_t n, Masks m) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t pos = (uint32_t)e[i];
    uint32_t d = 0;
    for (int k = 0; k < m.n; ++k) d |= valid1(m.v[k], pos) ? 0u : 1u;
    e[i] = ((uint64_t)d << 32) | pos;
  }
}

__global__ void count_kept_kernel(int64_t n, Masks m, unsigned long long* kept) {
  int64_t c = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    bool ok = true;
    for (int k = 0; k < m.n; ++k) ok = ok && valid1(m.v[k], i);
    c += ok ? 1 : 0;
  }
  c = warp_sum(c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(kept, (unsigned long long)c);
}

__global__ void perm_out_kernel(const uint64_t* e, int64_t n, int32_t* perm) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    perm[i] = (int32_t)(uint32_t)e[i];
}

// ------------------------------------------------------------------------------- segments
struct KeySet {
  nvtb_col_t c[kMaxKeys];
  int n;
};

struct BoundaryFlag {
  KeySet ks;
  const int32_t* perm;
  __device__ __forceinline__ int64_t operator()(int64_t i) const {
    if (i == 0) return 1;
    const int32_t a = perm[i - 1], b = perm[i];
    for (int k = 0; k < ks.n; ++k) {
      const bool va = valid1(ks.c[k].validity, a), vb = valid1(ks.c[k].validity, b);
      if (va != vb) return 1;
      if (va && sort_image(ks.c[k].data, ks.c[k].dtype, a) != sort_image(ks.c[k].data, ks.c[k].dtype, b)) return 1;
    }
    return 0;
  }
};

struct StartSink {
  int64_t* offsets;
  __device__ __forceinline__ void operator()(int64_t i, int64_t prefix, int64_t v) const {
    if (v) offsets[prefix] = i;
  }
};

__global__ void close_offsets_kernel(int64_t* offsets, const int64_t* n_groups, const int64_t* n_rows) {
  offsets[*n_groups] = *n_rows;
}

// --------------------------------------------------------------------------- segment aggs
enum { kCount = 0, kSum, kMean, kMin, kMax, kStd, kVar, kFirst, kLast, kNumAggs };

struct AggOut {
  void* out[kNumAggs];
  uint32_t* valid[kNumAggs];
};

__device__ __forceinline__ void set_valid(uint32_t* v, int64_t g) {
  if (v) atomicOr(v + (g >> 5), 1u << (g & 31));
}

struct LongAcc {
  double cnt, sum, sq;         // sums of (x - K), K = the group's first value
  unsigned long long mn, mx;   // images
};

template <typename T>
__device__ __forceinline__ void write_aggs(const AggOut& o, int64_t g, double cnt, double sumd, double sq, double K,
                                           uint64_t mn, uint64_t mx) {
  if (o.out[kCount]) reinterpret_cast<int32_t*>(o.out[kCount])[g] = (int32_t)cnt;
  if (o.out[kSum]) reinterpret_cast<float*>(o.out[kSum])[g] = (float)(cnt > 0 ? sumd + cnt * K : 0.0);
  if (o.out[kMean]) {
    reinterpret_cast<float*>(o.out[kMean])[g] = cnt > 0 ? (float)(K + sumd / cnt) : 0.0f;
    if (cnt > 0) set_valid(o.valid[kMean], g);
  }
  if (o.out[kMin]) {
    reinterpret_cast<T*>(o.out[kMin])[g] = cnt > 0 ? from_image<T>(mn) : (T)0;
    if (cnt > 0) set_valid(o.valid[kMin], g);
  }
  if (o.out[kMax]) {
    reinterpret_cast<T*>(o.out[kMax])[g] = cnt > 0 ? from_image<T>(mx) : (T)0;
    if (cnt > 0) set_valid(o.valid[kMax], g);
  }
  if (o.out[kVar] || o.out[kStd]) {
    double var = 0.0;
    if (cnt > 1) {
      var = (sq - sumd * sumd / cnt) / (cnt - 1.0);
      if (var < 0.0) var = 0.0;
    }
    if (o.out[kVar]) {
      reinterpret_cast<float*>(o.out[kVar])[g] = (float)var;
      if (cnt > 1) set_valid(o.valid[kVar], g);
    }
    if (o.out[kStd]) {
      reinterpret_cast<float*>(o.out[kStd])[g] = (float)sqrt(var);
      if (cnt > 1) set_valid(o.valid[kStd], g);
    }
  }
}

// the shift K of a group: its first row's value when that is valid, else 0 (same for every chunk)
template <typename T>
__device__ __forceinline__ double group_shift(const T* x, const uint8_t* valid, const int32_t* perm, int64_t start) {
  const int32_t p = perm[start];
  return valid1(valid, p) ? (double)x[p] : 0.0;
}

// one thread per group: first / last of every group, everything else of the short groups
template <typename T>
__global__ void __launch_bounds__(kGbThreads) seg_short_kernel(const T* __restrict__ x, const uint8_t* __restrict__ valid,
                                                               const int32_t* __restrict__ perm,
                                                               const int64_t* __restrict__ off, int64_t n_groups,
                                                               AggOut o, int need_stats) {
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = off[g], e = off[g + 1];
    if (o.out[kFirst]) {
      const int32_t p = perm[s];
      const bool ok = valid1(valid, p);
      reinterpret_cast<T*>(o.out[kFirst])[g] = ok ? x[p] : (T)0;
      if (ok) set_valid(o.valid[kFirst], g);
    }
    if (o.out[kLast]) {
      const int32_t p = perm[e - 1];
      const bool ok = valid1(valid, p);
      reinterpret_cast<T*>(o.out[kLast])[g] = ok ? x[p] : (T)0;
      if (ok) set_valid(o.valid[kLast], g);
    }
    if (!need_stats || e - s > kShortMax) continue;
    const double K = group_shift(x, valid, perm, s);
    double cnt = 0, sumd = 0, sq = 0;
    uint64_t mn = ~0ull, mx = 0ull;
    for (int64_t r = s; r < e; ++r) {
      const int32_t p = perm[r];
      if (!valid1(valid, p)) continue;
      const T v = x[p];
      const double d = (double)v - K;
      cnt += 1.0;
      sumd += d;
      sq += d * d;
      const uint64_t m = to_image<T>(v);
      mn = m < mn ? m : mn;
      mx = m > mx ? m : mx;
    }
    write_aggs<T>(o, g, cnt, sumd, sq, K, mn, mx);
  }
}

// chunk count of a group on the long path
struct ChunkCount {
  const int64_t* off;
  __device__ __forceinline__ int64_t operator()(int64_t g) const {
    const int64_t len = off[g + 1] - off[g];
    return len > kShortMax ? (len + kChunk - 1) / kChunk : 0;
  }
};

struct ChunkSink {
  int64_t* choff;
  LongAcc* acc;
  __device__ __forceinline__ void operator()(int64_t g, int64_t prefix, int64_t v) const {
    choff[g] = prefix;
    if (v) acc[g] = LongAcc{0.0, 0.0, 0.0, ~0ull, 0ull};
  }
};

template <typename T>
__global__ void __launch_bounds__(kGbThreads) seg_long_kernel(const T* __restrict__ x, const uint8_t* __restrict__ valid,
                                                              const int32_t* __restrict__ perm,
                                                              const int64_t* __restrict__ off,
                                                              const int64_t* __restrict__ choff, int64_t n_groups,
                                                              const int64_t* __restrict__ n_chunks, LongAcc* acc) {
  __shared__ double s_d[3][kGbThreads / 32];
  __shared__ unsigned long long s_m[2][kGbThreads / 32];
  __shared__ int64_t s_g;
  const int64_t total = *n_chunks;
  for (int64_t c = blockIdx.x; c < total; c += gridDim.x) {
    if (threadIdx.x == 0) {            // the group of chunk c: last g with choff[g] <= c
      int64_t lo = 0, hi = n_groups;
      while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (choff[mid] <= c) lo = mid; else hi = mid;
      }
      s_g = lo;
    }
    __syncthreads();
    const int64_t g = s_g;
    const int64_t s = off[g], e = off[g + 1];
    const int64_t r0 = s + (c - choff[g]) * kChunk;
    const int64_t r1 = r0 + kChunk < e ? r0 + kChunk : e;
    const double K = group_shift(x, valid, perm, s);
    double cnt = 0, sumd = 0, sq = 0;
    uint64_t mn = ~0ull, mx = 0ull;
    for (int64_t r = r0 + threadIdx.x; r < r1; r += kGbThreads) {
      const int32_t p = perm[r];
      if (!valid1(valid, p)) continue;
      const T v = x[p];
      const double d = (double)v - K;
      cnt += 1.0;
      sumd += d;
      sq += d * d;
      const uint64_t m = to_image<T>(v);
      mn = m < mn ? m : mn;
      mx = m > mx ? m : mx;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      cnt += __shfl_down_sync(0xFFFFFFFFu, cnt, o);
      sumd += __shfl_down_sync(0xFFFFFFFFu, sumd, o);
      sq += __shfl_down_sync(0xFFFFFFFFu, sq, o);
      const uint64_t a = __shfl_down_sync(0xFFFFFFFFu, mn, o), b = __shfl_down_sync(0xFFFFFFFFu, mx, o);
      mn = a < mn ? a : mn;
      mx = b > mx ? b : mx;
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
      s_d[0][w] = cnt; s_d[1][w] = sumd; s_d[2][w] = sq;
      s_m[0][w] = mn; s_m[1][w] = mx;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int k = 1; k < kGbThreads / 32; ++k) {
        cnt += s_d[0][k]; sumd += s_d[1][k]; sq += s_d[2][k];
        mn = s_m[0][k] < mn ? s_m[0][k] : mn;
        mx = s_m[1][k] > mx ? s_m[1][k] : mx;
      }
      if (cnt > 0) {
        atomicAdd(&acc[g].cnt, cnt);
        atomicAdd(&acc[g].sum, sumd);
        atomicAdd(&acc[g].sq, sq);
        atomicMin(&acc[g].mn, (unsigned long long)mn);
        atomicMax(&acc[g].mx, (unsigned long long)mx);
      }
    }
    __syncthreads();
  }
}

template <typename T>
__global__ void seg_long_finish_kernel(const T* __restrict__ x, const uint8_t* __restrict__ valid,
                                       const int32_t* __restrict__ perm, const int64_t* __restrict__ off,
                                       int64_t n_groups, const LongAcc* __restrict__ acc, AggOut o) {
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = off[g];
    if (off[g + 1] - s <= kShortMax) continue;
    const LongAcc a = acc[g];
    write_aggs<T>(o, g, a.cnt, a.sum, a.sq, group_shift(x, valid, perm, s), a.mn, a.mx);
  }
}

// --------------------------------------------------------------------- median / nunique
template <typename T>
struct DistinctFlag {            // row i (sorted) is valid and differs from row i-1
  const T* x;
  const uint8_t* valid;
  const int32_t* perm;
  __device__ __forceinline__ int64_t operator()(int64_t i) const {
    const int32_t p = perm[i];
    if (!valid1(valid, p)) return 0;
    if (i == 0) return 1;
    const int32_t q = perm[i - 1];
    return (!valid1(valid, q) || x[q] != x[p]) ? 1 : 0;
  }
};

struct PrefixSink {
  int64_t* pre;
  __device__ __forceinline__ void operator()(int64_t i, int64_t prefix, int64_t) const { pre[i] = prefix; }
};

template <typename T>
__global__ void seg_sorted_kernel(const T* __restrict__ x, const uint8_t* __restrict__ valid,
                                  const int32_t* __restrict__ perm, const int64_t* __restrict__ off, int64_t n_groups,
                                  int64_t n_rows, const int64_t* __restrict__ pre, const int64_t* __restrict__ total,
                                  float* median, uint32_t* median_valid, int32_t* nunique) {
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = off[g], e = off[g + 1];
    int64_t lo = s, hi = e;                    // first null row (nulls are last in the group)
    if (valid != nullptr) {
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (valid1(valid, perm[mid])) lo = mid + 1; else hi = mid;
      }
    } else {
      lo = e;
    }
    const int64_t c = lo - s;
    if (median) {
      if (c > 0) {
        const double a = (double)x[perm[s + (c - 1) / 2]], b = (double)x[perm[s + c / 2]];
        median[g] = (float)((a + b) * 0.5);
        set_valid(median_valid, g);
      } else {
        median[g] = 0.0f;
      }
    }
    if (nunique) {
      // the group's first valid row counts once; rows (s, s + c) count where they change value
      const int64_t pe = s + c < n_rows ? pre[s + c] : *total;
      const int64_t ps = s + 1 < n_rows ? pre[s + 1] : *total;
      nunique[g] = c > 0 ? (int32_t)(1 + pe - ps) : 0;
    }
  }
}

// ------------------------------------------------------------------------------- gathers
template <typename T>
__global__ void gather_rows_kernel(const T* __restrict__ src, const uint8_t* __restrict__ sv,
                                   const int32_t* __restrict__ perm, const int64_t* __restrict__ idx, int shift,
                                   int64_t n, T* __restrict__ out, uint32_t* __restrict__ ov) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t n32 = (n + 31) & ~(int64_t)31;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n32; i += stride) {
    bool ok = false;
    if (i < n) {
      int64_t r = idx ? idx[i] + shift : i;
      r = perm ? (int64_t)perm[r] : r;
      out[i] = src[r];
      ok = valid1(sv, r);
    }
    if (ov) {
      const unsigned b = __ballot_sync(0xFFFFFFFFu, ok);
      if ((threadIdx.x & 31) == 0) ov[i >> 5] = b;
    }
  }
}

// ------------------------------------------------------------------------------ list slice
struct SliceSpec {
  const int64_t* off;       // source offsets [rows + 1]
  const int32_t* perm;      // may be NULL
  const int64_t* idx;       // may be NULL
  int shift;
  int64_t start, end;
  int pad;
  int64_t max_elements;
  __device__ __forceinline__ int64_t src_row(int64_t r) const {
    int64_t s = idx ? idx[r] + shift : r;
    return perm ? (int64_t)perm[s] : s;
  }
  // Python slicing row[start:end] on a row of L elements -> (first element, length)
  __device__ __forceinline__ void bounds(int64_t L, int64_t* a, int64_t* len) const {
    int64_t lo = start < 0 ? L + start : start;
    int64_t hi = end < 0 ? L + end : end;
    lo = lo < 0 ? 0 : (lo > L ? L : lo);
    hi = hi < 0 ? 0 : (hi > L ? L : hi);
    *a = lo;
    *len = hi > lo ? hi - lo : 0;
    if (pad && *len > max_elements) *len = max_elements;
  }
};

struct SliceSize {
  SliceSpec sp;
  __device__ __forceinline__ int64_t operator()(int64_t r) const {
    if (sp.pad) return sp.max_elements;
    const int64_t s = sp.src_row(r);
    int64_t a, len;
    sp.bounds(sp.off[s + 1] - sp.off[s], &a, &len);
    return len;
  }
};

struct OffsetSink {
  int64_t* out;
  __device__ __forceinline__ void operator()(int64_t r, int64_t prefix, int64_t) const { out[r] = prefix; }
};

template <typename T>
__global__ void list_copy_kernel(SliceSpec sp, const T* __restrict__ leaves, const uint8_t* __restrict__ lv,
                                 int64_t n_rows, const int64_t* __restrict__ out_off, int64_t total, T pad_value,
                                 T* __restrict__ out, uint32_t* __restrict__ ov) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t n32 = (total + 31) & ~(int64_t)31;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n32; j += stride) {
    bool ok = false;
    if (j < total) {
      int64_t lo = 0, hi = n_rows;             // output row of element j: last r with out_off[r] <= j
      while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (out_off[mid] <= j) lo = mid; else hi = mid;
      }
      const int64_t r = lo, k = j - out_off[r];
      const int64_t s = sp.src_row(r);
      const int64_t base = sp.off[s];
      int64_t a, len;
      sp.bounds(sp.off[s + 1] - base, &a, &len);
      if (k < len) {
        out[j] = leaves[base + a + k];
        ok = valid1(lv, base + a + k);
      } else {
        out[j] = pad_value;
        ok = true;
      }
    }
    if (ov) {
      const unsigned b = __ballot_sync(0xFFFFFFFFu, ok);
      if ((threadIdx.x & 31) == 0) ov[j >> 5] = b;
    }
  }
}

}  // namespace
}  // namespace nvtb

using namespace nvtb;

extern "C" {

int nvtb_sort_rows(const nvtb_col_t* keys, const int* descending, int nkeys, int n_drop_null, int64_t n,
                   int32_t* perm_out, int64_t* n_kept_dev, void* stream) {
  NVTB_REQUIRE(keys != nullptr && nkeys >= 1 && nkeys <= kMaxKeys, "nkeys must be in [1, 8]");
  NVTB_REQUIRE(n_drop_null >= 0 && n_drop_null <= nkeys, "n_drop_null out of range");
  NVTB_REQUIRE(n >= 0 && n < ((int64_t)1 << 31), "nvtb_sort_rows orders fewer than 2^31 rows");
  NVTB_REQUIRE(n_kept_dev != nullptr, "NULL n_kept_dev");
  for (int k = 0; k < nkeys; ++k) {
    NVTB_REQUIRE(keys[k].dtype >= NVTB_I32 && keys[k].dtype <= NVTB_U8, "key dtype must be I32/I64/F32/F64/U8");
    NVTB_REQUIRE(n == 0 || keys[k].data != nullptr, "NULL key data");
  }
  cudaStream_t st = (cudaStream_t)stream;
  NVTB_CUDA_OK(cudaMemsetAsync(n_kept_dev, 0, sizeof(int64_t), st));
  if (n == 0) return NVTB_OK;
  NVTB_REQUIRE(perm_out != nullptr, "NULL perm_out");
  const int grid = gb_grid(n);

  // value ranges of every key (one synchronisation)
  unsigned long long* mm = nullptr;
  NVTB_CUDA_OK(cudaMallocAsync(&mm, sizeof(unsigned long long) * 2 * kMaxKeys, st));
  NVTB_CUDA_OK(cudaMemsetAsync(mm, 0xFF, sizeof(unsigned long long) * kMaxKeys, st));
  NVTB_CUDA_OK(cudaMemsetAsync(mm + kMaxKeys, 0, sizeof(unsigned long long) * kMaxKeys, st));
  for (int k = 0; k < nkeys; ++k) {
    key_range_kernel<<<grid, kGbThreads, 0, st>>>(keys[k], n, mm + k, mm + kMaxKeys + k);
    NVTB_LAUNCH_OK();
  }
  unsigned long long hmm[2 * kMaxKeys];
  NVTB_CUDA_OK(cudaMemcpyAsync(hmm, mm, sizeof(hmm), cudaMemcpyDeviceToHost, st));
  NVTB_CUDA_OK(cudaStreamSynchronize(st));
  NVTB_CUDA_OK(cudaFreeAsync(mm, st));

  uint64_t* a = nullptr;
  uint64_t* b = nullptr;
  void* scratch = nullptr;
  NVTB_CUDA_OK(cudaMallocAsync(&a, sizeof(uint64_t) * (size_t)n, st));
  NVTB_CUDA_OK(cudaMallocAsync(&b, sizeof(uint64_t) * (size_t)n, st));
  NVTB_CUDA_OK(cudaMallocAsync(&scratch, rx_scratch_bytes<uint64_t>(n, kRxMaxStableBits), st));
  NVTB_CUDA_OK(cudaMemsetAsync(scratch, 0, 256, st));
  identity_kernel<<<grid, kGbThreads, 0, st>>>(a, n);
  NVTB_LAUNCH_OK();

  auto sort_high = [&](int bits) -> int {
    int in_b = 0;
    int rc = rx_sort_bits<uint64_t>(a, b, nullptr, n, 32, 32 + bits, false, scratch, st, &in_b);
    if (rc) return rc;
    if (in_b) { uint64_t* t = a; a = b; b = t; }
    return NVTB_OK;
  };
  int rc = NVTB_OK;
  // least significant key first; within a key: value words, then (sort keys) its null flag
  for (int k = nkeys - 1; k >= 0 && rc == NVTB_OK; --k) {
    const uint64_t lo = hmm[k], hi = hmm[kMaxKeys + k];
    if (hi > lo) {                         // else: one value (or none) — nothing to order
      const uint64_t range = hi - lo;
      const int bits = 64 - __builtin_clzll(range);
      const int desc = descending && descending[k] ? 1 : 0;
      const uint64_t base = desc ? hi : lo;
      for (int shift = 0; shift < bits && rc == NVTB_OK; shift += 32) {
        set_digit_kernel<<<grid, kGbThreads, 0, st>>>(a, n, keys[k], base, desc, shift);
        NVTB_LAUNCH_OK();
        rc = sort_high(bits - shift < 32 ? bits - shift : 32);
      }
    }
    if (rc == NVTB_OK && k >= n_drop_null && keys[k].validity != nullptr) {
      Masks m{};
      m.v[0] = keys[k].validity;
      m.n = 1;
      set_null_digit_kernel<<<grid, kGbThreads, 0, st>>>(a, n, m);
      NVTB_LAUNCH_OK();
      rc = sort_high(1);
    }
  }
  Masks drop{};
  for (int k = 0; k < n_drop_null; ++k)
    if (keys[k].validity != nullptr) drop.v[drop.n++] = keys[k].validity;
  if (rc == NVTB_OK && drop.n > 0) {       // rows with a null group key go to the end, then are cut
    set_null_digit_kernel<<<grid, kGbThreads, 0, st>>>(a, n, drop);
    NVTB_LAUNCH_OK();
    rc = sort_high(1);
  }
  if (rc == NVTB_OK) {
    count_kept_kernel<<<grid, kGbThreads, 0, st>>>(n, drop, reinterpret_cast<unsigned long long*>(n_kept_dev));
    NVTB_LAUNCH_OK();
    perm_out_kernel<<<grid, kGbThreads, 0, st>>>(a, n, perm_out);
    NVTB_LAUNCH_OK();
  }
  NVTB_CUDA_OK(cudaFreeAsync(scratch, st));
  NVTB_CUDA_OK(cudaFreeAsync(a, st));
  NVTB_CUDA_OK(cudaFreeAsync(b, st));
  return rc;
}

int nvtb_segments(const nvtb_col_t* keys, int nkeys, const int32_t* perm, int64_t n_max, const int64_t* n_kept_dev,
                  int64_t* offsets_out, int64_t* n_groups_host, int64_t* n_kept_host, void* stream) {
  NVTB_REQUIRE(keys != nullptr && nkeys >= 1 && nkeys <= kMaxKeys, "nkeys must be in [1, 8]");
  NVTB_REQUIRE(n_max >= 0 && n_kept_dev && offsets_out && n_groups_host && n_kept_host, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  ScanScratch sc;
  int rc = scan_alloc(&sc, n_max, st);
  if (rc) return rc;
  BoundaryFlag f;
  f.ks.n = nkeys;
  for (int k = 0; k < nkeys; ++k) f.ks.c[k] = keys[k];
  f.perm = perm;
  rc = device_scan(f, StartSink{offsets_out}, n_kept_dev, n_max, sc, st);
  if (rc) return rc;
  close_offsets_kernel<<<1, 1, 0, st>>>(offsets_out, sc.total, n_kept_dev);
  NVTB_LAUNCH_OK();
  int64_t h[2];
  NVTB_CUDA_OK(cudaMemcpyAsync(&h[0], sc.total, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  NVTB_CUDA_OK(cudaMemcpyAsync(&h[1], n_kept_dev, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  NVTB_CUDA_OK(cudaFreeAsync(sc.total, st));
  NVTB_CUDA_OK(cudaStreamSynchronize(st));
  *n_groups_host = h[0];
  *n_kept_host = h[1];
  return NVTB_OK;
}

int nvtb_gather_rows(const nvtb_col_t* src, const int32_t* perm, const int64_t* idx, int idx_shift, int64_t n,
                     void* out, uint8_t* validity_out, void* stream) {
  NVTB_REQUIRE(src != nullptr && n >= 0, "NULL column or n < 0");
  if (n == 0) return NVTB_OK;
  NVTB_REQUIRE(src->data != nullptr && out != nullptr, "NULL data");
  NVTB_REQUIRE(src->validity == nullptr || validity_out != nullptr, "a column with nulls needs validity_out");
  NVTB_REQUIRE((reinterpret_cast<uintptr_t>(validity_out) & 3u) == 0, "validity_out must be 4-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  uint32_t* ov = src->validity ? reinterpret_cast<uint32_t*>(validity_out) : nullptr;
  const int grid = gb_grid(n);
  switch (dtype_size(src->dtype)) {
    case 1: gather_rows_kernel<uint8_t><<<grid, kGbThreads, 0, st>>>((const uint8_t*)src->data, src->validity, perm, idx, idx_shift, n, (uint8_t*)out, ov); break;
    case 4: gather_rows_kernel<uint32_t><<<grid, kGbThreads, 0, st>>>((const uint32_t*)src->data, src->validity, perm, idx, idx_shift, n, (uint32_t*)out, ov); break;
    case 8: gather_rows_kernel<uint64_t><<<grid, kGbThreads, 0, st>>>((const uint64_t*)src->data, src->validity, perm, idx, idx_shift, n, (uint64_t*)out, ov); break;
    default: NVTB_REQUIRE(false, "unsupported dtype");
  }
  NVTB_LAUNCH_OK();
  return NVTB_OK;
}

int nvtb_segment_agg(const nvtb_col_t* val, const int32_t* perm, const int64_t* offsets, int64_t n_groups,
                     void* const* out_host, uint8_t* const* validity_out_host, void* stream) {
  NVTB_REQUIRE(val != nullptr && out_host != nullptr && validity_out_host != nullptr && n_groups >= 0, "NULL argument");
  if (n_groups == 0) return NVTB_OK;
  NVTB_REQUIRE(val->data && perm && offsets, "NULL data / perm / offsets");
  cudaStream_t st = (cudaStream_t)stream;
  AggOut o;
  bool stats = false;
  const size_t vbytes = (size_t)((n_groups + 31) / 32) * 4;
  for (int a = 0; a < kNumAggs; ++a) {
    o.out[a] = out_host[a];
    o.valid[a] = reinterpret_cast<uint32_t*>(validity_out_host[a]);
    if (o.out[a] == nullptr) { o.valid[a] = nullptr; continue; }
    if (a != kFirst && a != kLast) stats = true;
    const bool needs = a == kMean || a == kMin || a == kMax || a == kStd || a == kVar ||
                       ((a == kFirst || a == kLast) && val->validity != nullptr);
    NVTB_REQUIRE(!needs || o.valid[a] != nullptr, "this aggregation needs a validity output");
    if (o.valid[a]) NVTB_CUDA_OK(cudaMemsetAsync(o.valid[a], 0, vbytes, st));
  }
  const int grid = gb_grid(n_groups);
  int rc = NVTB_OK;
  auto run = [&](auto tag) -> int {
    using T = decltype(tag);
    const T* x = reinterpret_cast<const T*>(val->data);
    seg_short_kernel<T><<<grid, kGbThreads, 0, st>>>(x, val->validity, perm, offsets, n_groups, o, stats ? 1 : 0);
    NVTB_LAUNCH_OK();
    if (!stats) return NVTB_OK;
    ScanScratch sc;
    int r = scan_alloc(&sc, n_groups, st);
    if (r) return r;
    int64_t* choff = nullptr;
    LongAcc* acc = nullptr;
    NVTB_CUDA_OK(cudaMallocAsync(&choff, sizeof(int64_t) * (size_t)n_groups, st));
    NVTB_CUDA_OK(cudaMallocAsync(&acc, sizeof(LongAcc) * (size_t)n_groups, st));
    r = device_scan(ChunkCount{offsets}, ChunkSink{choff, acc}, nullptr, n_groups, sc, st);
    if (r) return r;
    seg_long_kernel<T><<<sm_count() * 4, kGbThreads, 0, st>>>(x, val->validity, perm, offsets, choff, n_groups,
                                                              sc.total, acc);
    NVTB_LAUNCH_OK();
    seg_long_finish_kernel<T><<<grid, kGbThreads, 0, st>>>(x, val->validity, perm, offsets, n_groups, acc, o);
    NVTB_LAUNCH_OK();
    NVTB_CUDA_OK(cudaFreeAsync(acc, st));
    NVTB_CUDA_OK(cudaFreeAsync(choff, st));
    NVTB_CUDA_OK(cudaFreeAsync(sc.total, st));
    return NVTB_OK;
  };
  switch (val->dtype) {
    case NVTB_I32: rc = run(int32_t{}); break;
    case NVTB_I64: rc = run(int64_t{}); break;
    case NVTB_F32: rc = run(float{}); break;
    case NVTB_F64: rc = run(double{}); break;
    case NVTB_U8: rc = run(uint8_t{}); break;
    default: NVTB_REQUIRE(false, "unsupported value dtype");
  }
  return rc;
}

int nvtb_segment_sorted_agg(const nvtb_col_t* val, const int32_t* perm, const int64_t* offsets, int64_t n_groups,
                            int64_t n_rows, float* median_out, uint8_t* median_validity_out, int32_t* nunique_out,
                            void* stream) {
  NVTB_REQUIRE(val != nullptr && n_groups >= 0 && n_rows >= 0, "NULL column or negative size");
  NVTB_REQUIRE(median_out == nullptr || median_validity_out != nullptr, "median needs a validity output");
  if (n_groups == 0) return NVTB_OK;
  NVTB_REQUIRE(val->data && perm && offsets, "NULL data / perm / offsets");
  cudaStream_t st = (cudaStream_t)stream;
  if (median_validity_out)
    NVTB_CUDA_OK(cudaMemsetAsync(median_validity_out, 0, (size_t)((n_groups + 31) / 32) * 4, st));
  const int grid = gb_grid(n_groups);
  auto run = [&](auto tag) -> int {
    using T = decltype(tag);
    const T* x = reinterpret_cast<const T*>(val->data);
    ScanScratch sc;
    int r = scan_alloc(&sc, n_rows, st);
    if (r) return r;
    int64_t* pre = nullptr;
    if (nunique_out) {
      NVTB_CUDA_OK(cudaMallocAsync(&pre, sizeof(int64_t) * (size_t)(n_rows + 1), st));
      r = device_scan(DistinctFlag<T>{x, val->validity, perm}, PrefixSink{pre}, nullptr, n_rows, sc, st);
      if (r) return r;
    }
    seg_sorted_kernel<T><<<grid, kGbThreads, 0, st>>>(x, val->validity, perm, offsets, n_groups, n_rows, pre, sc.total,
                                                      median_out, reinterpret_cast<uint32_t*>(median_validity_out),
                                                      nunique_out);
    NVTB_LAUNCH_OK();
    if (pre) NVTB_CUDA_OK(cudaFreeAsync(pre, st));
    NVTB_CUDA_OK(cudaFreeAsync(sc.total, st));
    return NVTB_OK;
  };
  switch (val->dtype) {
    case NVTB_I32: return run(int32_t{});
    case NVTB_I64: return run(int64_t{});
    case NVTB_F32: return run(float{});
    case NVTB_F64: return run(double{});
    case NVTB_U8: return run(uint8_t{});
    default: NVTB_REQUIRE(false, "unsupported value dtype");
  }
  return NVTB_OK;
}

int nvtb_list_slice_offsets(const int64_t* offsets, int64_t n_rows, const int32_t* perm, const int64_t* idx,
                            int idx_shift, int64_t start, int64_t end, int pad, int64_t max_elements,
                            int64_t* offsets_out, int64_t* total_host, void* stream) {
  NVTB_REQUIRE(n_rows >= 0 && offsets_out != nullptr && total_host != nullptr, "NULL argument");
  NVTB_REQUIRE(!pad || max_elements >= 0, "padding needs a bounded slice");
  cudaStream_t st = (cudaStream_t)stream;
  *total_host = 0;
  if (n_rows == 0) {
    NVTB_CUDA_OK(cudaMemsetAsync(offsets_out, 0, sizeof(int64_t), st));
    return NVTB_OK;
  }
  NVTB_REQUIRE(offsets != nullptr, "NULL offsets");
  SliceSpec sp{offsets, perm, idx, idx_shift, start, end, pad ? 1 : 0, max_elements};
  ScanScratch sc;
  int rc = scan_alloc(&sc, n_rows, st);
  if (rc) return rc;
  rc = device_scan(SliceSize{sp}, OffsetSink{offsets_out}, nullptr, n_rows, sc, st);
  if (rc) return rc;
  NVTB_CUDA_OK(cudaMemcpyAsync(offsets_out + n_rows, sc.total, sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
  NVTB_CUDA_OK(cudaFreeAsync(sc.total, st));
  if (pad) {
    *total_host = n_rows * max_elements;
    return NVTB_OK;
  }
  int64_t t = 0;
  NVTB_CUDA_OK(cudaMemcpyAsync(&t, offsets_out + n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  NVTB_CUDA_OK(cudaStreamSynchronize(st));
  *total_host = t;
  return NVTB_OK;
}

int nvtb_list_slice(const int64_t* offsets, const nvtb_col_t* leaves, int64_t n_rows, const int32_t* perm,
                    const int64_t* idx, int idx_shift, int64_t start, int64_t end, int pad, int64_t max_elements,
                    double pad_value, const int64_t* offsets_out, int64_t total, void* leaves_out,
                    uint8_t* validity_out, void* stream) {
  NVTB_REQUIRE(leaves != nullptr && n_rows >= 0 && total >= 0, "NULL leaves or negative size");
  if (total == 0) return NVTB_OK;
  NVTB_REQUIRE(offsets && offsets_out && leaves_out, "NULL offsets / output");
  NVTB_REQUIRE(leaves->validity == nullptr || validity_out != nullptr, "leaves with nulls need validity_out");
  cudaStream_t st = (cudaStream_t)stream;
  SliceSpec sp{offsets, perm, idx, idx_shift, start, end, pad ? 1 : 0, max_elements};
  uint32_t* ov = leaves->validity ? reinterpret_cast<uint32_t*>(validity_out) : nullptr;
  const int grid = gb_grid(total);
  switch (leaves->dtype) {
    case NVTB_I32: list_copy_kernel<int32_t><<<grid, kGbThreads, 0, st>>>(sp, (const int32_t*)leaves->data, leaves->validity, n_rows, offsets_out, total, (int32_t)pad_value, (int32_t*)leaves_out, ov); break;
    case NVTB_I64: list_copy_kernel<int64_t><<<grid, kGbThreads, 0, st>>>(sp, (const int64_t*)leaves->data, leaves->validity, n_rows, offsets_out, total, (int64_t)pad_value, (int64_t*)leaves_out, ov); break;
    case NVTB_F32: list_copy_kernel<float><<<grid, kGbThreads, 0, st>>>(sp, (const float*)leaves->data, leaves->validity, n_rows, offsets_out, total, (float)pad_value, (float*)leaves_out, ov); break;
    case NVTB_F64: list_copy_kernel<double><<<grid, kGbThreads, 0, st>>>(sp, (const double*)leaves->data, leaves->validity, n_rows, offsets_out, total, pad_value, (double*)leaves_out, ov); break;
    case NVTB_U8: list_copy_kernel<uint8_t><<<grid, kGbThreads, 0, st>>>(sp, (const uint8_t*)leaves->data, leaves->validity, n_rows, offsets_out, total, (uint8_t)pad_value, (uint8_t*)leaves_out, ov); break;
    default: NVTB_REQUIRE(false, "unsupported leaf dtype");
  }
  NVTB_LAUNCH_OK();
  return NVTB_OK;
}

}  // extern "C"
