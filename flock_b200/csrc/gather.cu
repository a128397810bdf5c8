// gather.cu -- row gather through an index vector: the arrow `take` kernel of the reference's
// HashJoinExec output construction and RepartitionExec (call shape in
// playground/src/distributed_plan/shuffle_writer.rs:129-146), and the Utf8 half of `filter`.
//
//   fixed width : out[i] = in[idx[i]]
//   Utf8        : lengths -> exclusive scan (single pass, the grid-wide prefix of compact.cuh) -> byte copy where each
//                 warp owns 32 consecutive OUTPUT rows, so output bytes are written densely in order.
#include <algorithm>

#include "compact.cuh"
#include "device_utils.cuh"
#include "internal.h"

namespace fg {

constexpr int GA_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(GA_THREADS) gather_fixed_kernel(const T* __restrict__ in, const uint32_t* __restrict__ idx,
                                                                   T* __restrict__ out, int64_t n) {
  const int64_t stride = int64_t(gridDim.x) * GA_THREADS;
  int64_t i = int64_t(blockIdx.x) * GA_THREADS + threadIdx.x;
  // 4 independent gathers in flight per thread
  for (; i + 3 * stride < n; i += 4 * stride) {
    uint32_t a = idx[i], b = idx[i + stride], c = idx[i + 2 * stride], d = idx[i + 3 * stride];
    T va = in[a], vb = in[b], vc = in[c], vd = in[d];
    out[i] = va;
    out[i + stride] = vb;
    out[i + 2 * stride] = vc;
    out[i + 3 * stride] = vd;
  }
  for (; i < n; i += stride) out[i] = in[idx[i]];
}

// All fixed-width columns of one take() in ONE launch: the index is read once per row, the gathers of a row's columns
// are independent and in flight together (q3's join output: 4 launches -> 1).
constexpr int GM_MAX_COLS = 16;
constexpr int kGatherTotalsSlot = 384;  // d_scalars[384 .. 447]: byte totals of the Utf8 columns of one take()
struct GatherMultiArgs {
  const uint32_t* idx;
  int64_t n;
  int32_t n_cols;
  int32_t pad;
  const void* src[GM_MAX_COLS];
  void* dst[GM_MAX_COLS];
  int32_t width[GM_MAX_COLS];
};

// PAD: the index may hold the pad sentinel GATHER_PAD (an outer join's unmatched row): its value is 0.  The Inner join
// and every other take() launch PAD = false, which is the kernel as it was before the sentinel existed.
constexpr uint32_t GATHER_PAD = ~0u;

template <bool PAD>
__global__ void __launch_bounds__(GA_THREADS) gather_fixed_multi_kernel(const __grid_constant__ GatherMultiArgs a) {
  const int64_t stride = int64_t(gridDim.x) * GA_THREADS;
  for (int64_t i = int64_t(blockIdx.x) * GA_THREADS + threadIdx.x; i < a.n; i += 2 * stride) {
    const int64_t j = i + stride;
    const uint32_t r0 = a.idx[i], r1 = j < a.n ? a.idx[j] : (PAD ? GATHER_PAD : 0u);
    for (int c = 0; c < a.n_cols; ++c) {
      if (a.width[c] == 4) {
        const uint32_t v0 = PAD && r0 == GATHER_PAD ? 0u : static_cast<const uint32_t*>(a.src[c])[r0];
        const uint32_t v1 = PAD && r1 == GATHER_PAD ? 0u : j < a.n ? static_cast<const uint32_t*>(a.src[c])[r1] : 0u;
        static_cast<uint32_t*>(a.dst[c])[i] = v0;
        if (j < a.n) static_cast<uint32_t*>(a.dst[c])[j] = v1;
      } else {
        const uint64_t v0 = PAD && r0 == GATHER_PAD ? 0ull : static_cast<const uint64_t*>(a.src[c])[r0];
        const uint64_t v1 = PAD && r1 == GATHER_PAD ? 0ull : j < a.n ? static_cast<const uint64_t*>(a.src[c])[r1] : 0ull;
        static_cast<uint64_t*>(a.dst[c])[i] = v0;
        if (j < a.n) static_cast<uint64_t*>(a.dst[c])[j] = v1;
      }
    }
  }
}

// Validity of a column taken through an index with pad sentinels: 0 for a sentinel, else the source's byte (1 when the
// source has no validity).
__global__ void __launch_bounds__(GA_THREADS) gather_valid_pad_kernel(const uint8_t* __restrict__ in, const uint32_t* __restrict__ idx,
                                                                      uint8_t* __restrict__ out, int64_t n) {
  const int64_t stride = int64_t(gridDim.x) * GA_THREADS;
  for (int64_t i = int64_t(blockIdx.x) * GA_THREADS + threadIdx.x; i < n; i += stride) {
    const uint32_t r = idx[i];
    out[i] = r == GATHER_PAD ? uint8_t(0) : in ? in[r] : uint8_t(1);
  }
}

// ---- Utf8 pass 1: out_off[i] = sum_{j<i} len(idx[j]); out_off[n] = total ---------------------------
constexpr int GL_ITEMS = 8;
constexpr int GL_TILE = GA_THREADS * GL_ITEMS;

struct GatherLenArgs {
  const int32_t* in_off;
  const uint32_t* idx;  // may be NULL: identity (plain offsets rebuild)
  int32_t* out_off;
  int64_t n;
  CompactScratch sc;  // grid-wide exclusive prefix of the tiles' byte counts (compact.cuh); sc.out_count = total bytes
};

template <bool PAD>
__global__ void __launch_bounds__(GA_THREADS) gather_lengths_scan_kernel(const __grid_constant__ GatherLenArgs a) {
  __shared__ CompactSmem<1, 16> sm;
  __shared__ unsigned long long s_warp[GA_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  long long tile;
  for (int it = 0; (tile = cp_next_tile(sm, a.sc, it)) >= 0; ++it) {
    const int64_t i0 = tile * GL_TILE + int64_t(tid) * GL_ITEMS;
    unsigned len[GL_ITEMS];
    unsigned long long local = 0;
#pragma unroll
    for (int k = 0; k < GL_ITEMS; ++k) {
      len[k] = 0;
      if (i0 + k < a.n) {
        int64_t r = a.idx ? int64_t(a.idx[i0 + k]) : i0 + k;
        if (!PAD || r != int64_t(GATHER_PAD)) len[k] = unsigned(a.in_off[r + 1] - a.in_off[r]);
      }
      local += len[k];
    }
    unsigned long long incl = warp_inclusive_sum(local);
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned long long warp_base = 0, tile_total = 0;
#pragma unroll
    for (int w = 0; w < GA_THREADS / 32; ++w) {
      unsigned long long v = s_warp[w];
      if (w < warp) warp_base += v;
      tile_total += v;
    }
    if (a.sc.single_wave) cp_grid_prefix(sm, a.sc, tile, tile_total);
    else cp_block_lookback(sm, a.sc, tile, tile_total);
    unsigned long long run = sm.excl + warp_base + (incl - local);
#pragma unroll
    for (int k = 0; k < GL_ITEMS; ++k) {
      if (i0 + k < a.n) a.out_off[i0 + k] = int32_t(run);
      run += len[k];
    }
    if (tile == a.sc.num_tiles - 1 && tid == 0) a.out_off[a.n] = int32_t(sm.excl + tile_total);
    __syncthreads();  // sm / s_warp are reused by the next tile
  }
}

// All Utf8 columns of one take() in ONE single-wave launch: CTA b scans tile b % tiles of column b / tiles; the
// columns' prefixes are independent groups of the shared count words (compact.cuh: cp_grid_prefix group_base).
constexpr int GL_MAX_COLS = 8;
struct GatherLenMultiArgs {
  const int32_t* in_off[GL_MAX_COLS];
  int32_t* out_off[GL_MAX_COLS];
  unsigned long long* totals;  // [n_cols] byte totals
  const uint32_t* idx;
  int64_t n;
  int32_t n_cols, tiles;       // tiles per column
  CompactScratch sc;           // sc.num_tiles = n_cols * tiles, single wave
};

template <bool PAD>
__global__ void __launch_bounds__(GA_THREADS) gather_lengths_scan_multi_kernel(const __grid_constant__ GatherLenMultiArgs a) {
  __shared__ CompactSmem<1, 16> sm;
  __shared__ unsigned long long s_warp[GA_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int col = int(blockIdx.x) / a.tiles;
  const long long tile = int(blockIdx.x) % a.tiles;
  if (col >= a.n_cols) return;
  const int32_t* in_off = a.in_off[col];
  int32_t* out_off = a.out_off[col];
  const int64_t i0 = tile * GL_TILE + int64_t(tid) * GL_ITEMS;
  unsigned len[GL_ITEMS];
  unsigned long long local = 0;
#pragma unroll
  for (int k = 0; k < GL_ITEMS; ++k) {
    len[k] = 0;
    if (i0 + k < a.n) {
      const int64_t r = a.idx ? int64_t(a.idx[i0 + k]) : i0 + k;
      if (!PAD || r != int64_t(GATHER_PAD)) len[k] = unsigned(in_off[r + 1] - in_off[r]);
    }
    local += len[k];
  }
  const unsigned long long incl = warp_inclusive_sum(local);
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  unsigned long long warp_base = 0, tile_total = 0;
#pragma unroll
  for (int w = 0; w < GA_THREADS / 32; ++w) {
    const unsigned long long v = s_warp[w];
    if (w < warp) warp_base += v;
    tile_total += v;
  }
  cp_grid_prefix(sm, a.sc, tile, tile_total, (long long)col * a.tiles, tile == a.tiles - 1 ? 1 : 0, a.totals + col);
  unsigned long long run = sm.excl + warp_base + (incl - local);
#pragma unroll
  for (int k = 0; k < GL_ITEMS; ++k) {
    if (i0 + k < a.n) out_off[i0 + k] = int32_t(run);
    run += len[k];
  }
  if (tile == a.tiles - 1 && tid == 0) out_off[a.n] = int32_t(sm.excl + tile_total);
}

// ---- Utf8 pass 2: byte copy, one warp per 32 output rows -------------------------------------------
struct GatherCopyMultiArgs {
  const uint8_t* in_data[GL_MAX_COLS];
  const int32_t* in_off[GL_MAX_COLS];
  const int32_t* out_off[GL_MAX_COLS];
  uint8_t* out_data[GL_MAX_COLS];
  const uint32_t* idx;
  int64_t n;
};
constexpr int GU_STAGE = 2048;  // bytes of shared staging per warp

template <bool PAD>
__device__ __forceinline__ void gather_utf8_copy_body(const uint8_t* __restrict__ in_data, const int32_t* __restrict__ in_off,
                                                      const uint32_t* __restrict__ idx, const int32_t* __restrict__ out_off,
                                                      uint8_t* __restrict__ out_data, int64_t n) {
  // A warp owns 32 consecutive OUTPUT rows = one contiguous output byte range [d0, d1).  Each lane copies its own row
  // into the warp's shared staging area (laid out like the output, including its misalignment), then the warp writes
  // the range with aligned 4-byte stores.  NEXMark strings are short (names ~12 B, cities ~9 B): the earlier
  // byte-per-lane loop with a 5-step shuffle search per byte cost ~25 instructions per byte (0.5 TB/s on q8's names).
  __shared__ __align__(16) uint8_t s_stage[GA_THREADS / 32][GU_STAGE + 8];
  const int lane = threadIdx.x & 31;
  uint8_t* stage = s_stage[threadIdx.x >> 5];
  const int64_t warps_total = (int64_t(gridDim.x) * GA_THREADS) >> 5;
  const int64_t chunks = (n + 31) >> 5;
  for (int64_t chunk = (int64_t(blockIdx.x) * GA_THREADS + threadIdx.x) >> 5; chunk < chunks; chunk += warps_total) {
    const int64_t r0 = chunk << 5;
    const int rows = (n - r0) < 32 ? int(n - r0) : 32;
    int32_t dst_start = 0x7fffffff, src_start = 0, len = 0;
    if (lane < rows) {
      dst_start = out_off[r0 + lane];
      len = out_off[r0 + lane + 1] - dst_start;
      int64_t r = idx ? int64_t(idx[r0 + lane]) : r0 + lane;
      if (!PAD || r != int64_t(GATHER_PAD)) src_start = in_off[r];  // a padded row has length 0: no byte is read
    }
    const int32_t d0 = __shfl_sync(FULL_MASK, dst_start, 0);
    const int32_t d1 = out_off[r0 + rows];
    const int32_t total = d1 - d0, mis = d0 & 3;
    if (mis + total <= GU_STAGE) {
      if (len > 0) {
        uint8_t* mine = stage + mis + (dst_start - d0);
        const uint8_t* src = in_data + src_start;
        for (int32_t j = 0; j < len; ++j) mine[j] = src[j];
      }
      __syncwarp();
      uint8_t* out_base = out_data + (d0 - mis);  // 4-byte aligned (column buffers are 256-byte aligned)
      const int32_t n_words = (mis + total + 3) >> 2;
      for (int32_t w = lane; w < n_words; w += 32) {
        const int32_t lo = w << 2;
        if (lo >= mis && lo + 4 <= mis + total) {
          *reinterpret_cast<uint32_t*>(out_base + lo) = *reinterpret_cast<const uint32_t*>(stage + lo);
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (lo + e >= mis && lo + e < mis + total) out_base[lo + e] = stage[lo + e];
        }
      }
      __syncwarp();  // the staging area is reused by the next chunk
      continue;
    }
    // long strings: byte-per-lane copy; the owning row of a byte is found by a 5-step search over the warp's starts
    for (int32_t b0 = d0; b0 < d1; b0 += 32) {
      const int32_t b = b0 + lane;
      int lo = 0;
#pragma unroll
      for (int step = 16; step >= 1; step >>= 1) {
        int cand = lo + step;
        int32_t ds = __shfl_sync(FULL_MASK, dst_start, cand & 31);
        if (cand < rows && ds <= b) lo = cand;
      }
      const int32_t ds = __shfl_sync(FULL_MASK, dst_start, lo);
      const int32_t ss = __shfl_sync(FULL_MASK, src_start, lo);
      if (b < d1) out_data[b] = in_data[ss + (b - ds)];
    }
  }
}

template <bool PAD>
__global__ void __launch_bounds__(GA_THREADS) gather_utf8_copy_kernel(const uint8_t* __restrict__ in_data, const int32_t* __restrict__ in_off,
                                                                       const uint32_t* __restrict__ idx, const int32_t* __restrict__ out_off,
                                                                       uint8_t* __restrict__ out_data, int64_t n) {
  gather_utf8_copy_body<PAD>(in_data, in_off, idx, out_off, out_data, n);
}

// every Utf8 column of a take() in one launch: blockIdx.y = column
template <bool PAD>
__global__ void __launch_bounds__(GA_THREADS) gather_utf8_copy_multi_kernel(const __grid_constant__ GatherCopyMultiArgs a) {
  const int c = blockIdx.y;
  gather_utf8_copy_body<PAD>(a.in_data[c], a.in_off[c], a.idx, a.out_off[c], a.out_data[c], a.n);
}

// ------------------------------------------------------------------------------------------------
static int stream_grid(const CtxPtr& ctx, int64_t items, int per_block, int blocks_per_sm) {
  int64_t g = (items + per_block - 1) / per_block;
  return int(std::max<int64_t>(1, std::min<int64_t>(g, int64_t(ctx->sm_count) * blocks_per_sm)));
}

static int stream_grid(const CtxPtr& ctx, int64_t items, int per_block, int blocks_per_sm = 8);
// the validity bytes of a taken column: one more 1-byte gather
static void gather_validity(const CtxPtr& ctx, const Column& in, Column& out, const uint32_t* d_idx, int64_t n) {
  if (!in.validity) return;
  out.validity = alloc(ctx, size_t(n));
  if (n > 0) {
    {
      LaunchTimer lt(ctx, "gather_fixed_kernel<uint8_t>");
      gather_fixed_kernel<uint8_t><<<stream_grid(ctx, n, GA_THREADS * 4), GA_THREADS, 0, ctx->stream>>>(in.valid(), d_idx, out.validity->as<uint8_t>(), n);
    }
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);
  }
}

static Column gather_column_values(const CtxPtr& ctx, const Column& in, const uint32_t* d_idx, int64_t n);

Column gather_column(const CtxPtr& ctx, const Column& in, const uint32_t* d_idx, int64_t n) {
  Column out = gather_column_values(ctx, in, d_idx, n);
  gather_validity(ctx, in, out, d_idx, n);
  return out;
}

static Column gather_column_values(const CtxPtr& ctx, const Column& in, const uint32_t* d_idx, int64_t n) {
  FG_CHECK(!in.all_null, FLOCKGPU_ERR_UNSUPPORTED, "gather: NULL column \"%s\"", in.name.c_str());
  Column out;
  out.dtype = in.dtype;
  out.name = in.name;
  out.format = in.format;
  out.nullable = in.nullable;
  out.length = n;
  if (in.dtype != FLOCKGPU_UTF8) {
    int w = in.width();
    out.data = alloc(ctx, size_t(n) * w);
    if (n > 0) {
      int grid = stream_grid(ctx, n, GA_THREADS * 4);
      if (w == 4)
        {
          LaunchTimer lt(ctx, "gather_fixed_kernel<uint32_t>");
          gather_fixed_kernel<uint32_t><<<grid, GA_THREADS, 0, ctx->stream>>>(static_cast<const uint32_t*>(in.values()), d_idx,
                                                                            out.data->as<uint32_t>(), n);
        }
      else
        {
          LaunchTimer lt(ctx, "gather_fixed_kernel<uint64_t>");
          gather_fixed_kernel<uint64_t><<<grid, GA_THREADS, 0, ctx->stream>>>(static_cast<const uint64_t*>(in.values()), d_idx,
                                                                            out.data->as<uint64_t>(), n);
        }
      FG_CUDA(cudaGetLastError());
      count_launch(ctx);
    }
    return out;
  }
  out.offsets = alloc(ctx, size_t(n + 1) * 4);
  if (n == 0) {
    FG_CUDA(cudaMemsetAsync(out.offsets->ptr, 0, 4, ctx->stream));
    out.data = alloc(ctx, 0);
    out.values_bytes = 0;
    return out;
  }
  GatherLenArgs a{};
  a.in_off = in.offs();
  a.idx = d_idx;
  a.out_off = out.offsets->as<int32_t>();
  a.n = n;
  const int64_t num_tiles = (n + GL_TILE - 1) / GL_TILE;
  {
    a.sc = prepare_compact(ctx, num_tiles, resident_ctas(ctx, reinterpret_cast<const void*>(gather_lengths_scan_kernel<false>), GA_THREADS), ctx->d_scalars + 1);
    {
      LaunchTimer lt(ctx, "gather_lengths_scan_kernel");
      launch_compact(ctx, gather_lengths_scan_kernel<false>, a.sc, a);
    }
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);
  }
  unsigned long long total = 0;
  read_scalars(ctx, 1, 1, &total);
  FG_CHECK(total < (1ull << 31), FLOCKGPU_ERR_UNSUPPORTED, "gather: Utf8 result column \"%s\" exceeds 2^31-1 bytes", in.name.c_str());
  out.values_bytes = int64_t(total);
  out.data = alloc(ctx, size_t(total));
  if (total > 0) {
    int grid = stream_grid(ctx, (n + 31) / 32, GA_THREADS / 32);
    {
      LaunchTimer lt(ctx, "gather_utf8_copy_kernel");
      gather_utf8_copy_kernel<false><<<grid, GA_THREADS, 0, ctx->stream>>>(static_cast<const uint8_t*>(in.values()), in.offs(), d_idx,
                                                                  out.offsets->as<int32_t>(), out.data->as<uint8_t>(), n);
    }
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);
  }
  return out;
}

// take() of several columns through one index vector: one launch for all fixed-width columns; the Utf8 columns' length
// scans are launched back to back and their byte totals read with ONE host round trip (each used to cost its own).
// `pad` selects the PAD flavour of every kernel (see gather_fixed_multi_kernel); the launch labels say so, so a launch
// profile tells the outer join's takes from the Inner join's.
static std::vector<Column> gather_columns_values(const CtxPtr& ctx, const std::vector<const Column*>& in, const uint32_t* d_idx, int64_t n, bool pad);

// the validity of a padded take(): every column gets one (a padded row is NULL), one launch per column
static void gather_validity_pad(const CtxPtr& ctx, const Column& in, Column& out, const uint32_t* d_idx, int64_t n) {
  out.validity = alloc(ctx, size_t(n));
  out.nullable = true;
  if (n > 0) {
    {
      LaunchTimer lt(ctx, "gather_valid_pad_kernel");
      gather_valid_pad_kernel<<<stream_grid(ctx, n, GA_THREADS * 4), GA_THREADS, 0, ctx->stream>>>(in.valid(), d_idx, out.validity->as<uint8_t>(), n);
    }
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);
  }
}

std::vector<Column> null_columns(const CtxPtr& ctx, const Table& t, int64_t n) {
  std::vector<Column> out(t.cols.size());
  for (size_t k = 0; k < t.cols.size(); ++k) {
    const Column& c = t.cols[k];
    Column& o = out[k];
    o.dtype = c.dtype;
    o.name = c.name;
    o.format = c.format;
    o.nullable = true;
    o.length = n;
    o.validity = alloc(ctx, size_t(n));
    if (n > 0) FG_CUDA(cudaMemsetAsync(o.validity->ptr, 0, size_t(n), ctx->stream));
    if (c.dtype == FLOCKGPU_UTF8) {
      o.offsets = alloc(ctx, size_t(n + 1) * 4);
      FG_CUDA(cudaMemsetAsync(o.offsets->ptr, 0, size_t(n + 1) * 4, ctx->stream));
      o.data = alloc(ctx, 0);
      o.values_bytes = 0;
    } else {
      o.data = alloc(ctx, size_t(n) * c.width());
      if (n > 0) FG_CUDA(cudaMemsetAsync(o.data->ptr, 0, size_t(n) * c.width(), ctx->stream));
    }
  }
  return out;
}

std::vector<Column> gather_columns(const CtxPtr& ctx, const std::vector<const Column*>& in, const uint32_t* d_idx, int64_t n, bool pad) {
  if (pad) {
    // a column that is NULL as a whole (global aggregate over empty input) is NULL in every taken row too
    std::vector<const Column*> live;
    for (const Column* c : in)
      if (!c->all_null) live.push_back(c);
    std::vector<Column> got = gather_columns_values(ctx, live, d_idx, n, true);
    std::vector<Column> out;
    size_t g = 0;
    for (const Column* c : in) {
      if (c->all_null) {
        Table one;
        one.cols.push_back(*c);
        out.push_back(std::move(null_columns(ctx, one, n)[0]));
        continue;
      }
      gather_validity_pad(ctx, *c, got[g], d_idx, n);
      out.push_back(std::move(got[g++]));
    }
    return out;
  }
  std::vector<Column> out = gather_columns_values(ctx, in, d_idx, n, false);
  for (size_t k = 0; k < in.size(); ++k) gather_validity(ctx, *in[k], out[k], d_idx, n);
  return out;
}

static std::vector<Column> gather_columns_values(const CtxPtr& ctx, const std::vector<const Column*>& in, const uint32_t* d_idx, int64_t n, bool pad) {
  std::vector<Column> out(in.size());
  std::vector<size_t> fixed, utf8;
  for (size_t k = 0; k < in.size(); ++k) {
    const Column& c = *in[k];
    FG_CHECK(!c.all_null, FLOCKGPU_ERR_UNSUPPORTED, "gather: NULL column \"%s\"", c.name.c_str());
    Column& o = out[k];
    o.dtype = c.dtype;
    o.name = c.name;
    o.format = c.format;
    o.nullable = c.nullable;
    o.length = n;
    (c.dtype == FLOCKGPU_UTF8 ? utf8 : fixed).push_back(k);
  }
  const auto lengths_scan = pad ? gather_lengths_scan_kernel<true> : gather_lengths_scan_kernel<false>;
  const auto lengths_scan_multi = pad ? gather_lengths_scan_multi_kernel<true> : gather_lengths_scan_multi_kernel<false>;
  const auto copy = pad ? gather_utf8_copy_kernel<true> : gather_utf8_copy_kernel<false>;
  const auto copy_multi = pad ? gather_utf8_copy_multi_kernel<true> : gather_utf8_copy_multi_kernel<false>;
  for (size_t first = 0; first < fixed.size(); first += GM_MAX_COLS) {
    GatherMultiArgs a{};
    a.idx = d_idx;
    a.n = n;
    a.n_cols = int(std::min<size_t>(GM_MAX_COLS, fixed.size() - first));
    for (int c = 0; c < a.n_cols; ++c) {
      const Column& src = *in[fixed[first + c]];
      Column& o = out[fixed[first + c]];
      o.data = alloc(ctx, size_t(n) * src.width());
      a.src[c] = src.values();
      a.dst[c] = o.data->ptr;
      a.width[c] = src.width();
    }
    if (n > 0) {
      {
        LaunchTimer lt(ctx, pad ? "gather_fixed_multi_kernel<PAD>" : "gather_fixed_multi_kernel");
        (pad ? gather_fixed_multi_kernel<true> : gather_fixed_multi_kernel<false>)<<<stream_grid(ctx, n, GA_THREADS * 2), GA_THREADS, 0, ctx->stream>>>(a);
      }
      FG_CUDA(cudaGetLastError());
      count_launch(ctx);
    }
  }
  if (utf8.empty()) return out;
  FG_CHECK(utf8.size() <= 64, FLOCKGPU_ERR_UNSUPPORTED, "gather: more than 64 Utf8 columns");
  // ---- several Utf8 columns whose length scans fit ONE wave together: one scan launch, one host round trip for the
  // byte totals, one copy launch (q3's join output takes name, city and state: 6 launches -> 2)
  if (n > 0 && utf8.size() >= 2 && utf8.size() <= size_t(GL_MAX_COLS) && ctx->compact_mode == 0) {
    const int64_t tiles = (n + GL_TILE - 1) / GL_TILE;
    const int64_t resident = resident_ctas(ctx, reinterpret_cast<const void*>(lengths_scan_multi), GA_THREADS);
    if (tiles * int64_t(utf8.size()) <= resident) {
      GatherLenMultiArgs la{};
      la.idx = d_idx;
      la.n = n;
      la.n_cols = int(utf8.size());
      la.tiles = int(tiles);
      la.totals = ctx->d_scalars + kGatherTotalsSlot;
      for (size_t u = 0; u < utf8.size(); ++u) {
        Column& o = out[utf8[u]];
        o.offsets = alloc(ctx, size_t(n + 1) * 4);
        la.in_off[u] = in[utf8[u]]->offs();
        la.out_off[u] = o.offsets->as<int32_t>();
      }
      la.sc = prepare_compact(ctx, tiles * int64_t(utf8.size()), resident, ctx->d_scalars + kGatherTotalsSlot);
      if (la.sc.single_wave) {
        {
          LaunchTimer lt(ctx, pad ? "gather_lengths_scan_multi_kernel<PAD>" : "gather_lengths_scan_multi_kernel");
          launch_compact(ctx, lengths_scan_multi, la.sc, la);
        }
        FG_CUDA(cudaGetLastError());
        count_launch(ctx);
        std::vector<unsigned long long> totals(utf8.size());
        read_scalars(ctx, kGatherTotalsSlot, int(utf8.size()), totals.data());
        GatherCopyMultiArgs ca{};
        ca.idx = d_idx;
        ca.n = n;
        bool any = false;
        for (size_t u = 0; u < utf8.size(); ++u) {
          const Column& src = *in[utf8[u]];
          Column& o = out[utf8[u]];
          FG_CHECK(totals[u] < (1ull << 31), FLOCKGPU_ERR_UNSUPPORTED, "gather: Utf8 result column \"%s\" exceeds 2^31-1 bytes", src.name.c_str());
          o.values_bytes = int64_t(totals[u]);
          o.data = alloc(ctx, size_t(totals[u]));
          ca.in_data[u] = static_cast<const uint8_t*>(src.values());
          ca.in_off[u] = src.offs();
          ca.out_off[u] = o.offsets->as<int32_t>();
          ca.out_data[u] = o.data->as<uint8_t>();
          any |= totals[u] > 0;
        }
        if (any) {
          dim3 grid(unsigned(stream_grid(ctx, (n + 31) / 32, GA_THREADS / 32, 8 / int(utf8.size()) + 1)), unsigned(utf8.size()));
          {
            LaunchTimer lt(ctx, pad ? "gather_utf8_copy_multi_kernel<PAD>" : "gather_utf8_copy_multi_kernel");
            copy_multi<<<grid, GA_THREADS, 0, ctx->stream>>>(ca);
          }
          FG_CUDA(cudaGetLastError());
          count_launch(ctx);
        }
        return out;
      }
      // (prepare_compact chose look-back after all: fall through to the column-by-column path; the offsets buffers
      // allocated above are simply replaced)
    }
  }
  for (size_t u = 0; u < utf8.size(); ++u) {
    Column& o = out[utf8[u]];
    o.offsets = alloc(ctx, size_t(n + 1) * 4);
    if (n == 0) {
      FG_CUDA(cudaMemsetAsync(o.offsets->ptr, 0, 4, ctx->stream));
      o.data = alloc(ctx, 0);
      o.values_bytes = 0;
      continue;
    }
    GatherLenArgs a{};
    a.in_off = in[utf8[u]]->offs();
    a.idx = d_idx;
    a.out_off = o.offsets->as<int32_t>();
    a.n = n;
    const int64_t num_tiles = (n + GL_TILE - 1) / GL_TILE;
    a.sc = prepare_compact(ctx, num_tiles, resident_ctas(ctx, reinterpret_cast<const void*>(lengths_scan), GA_THREADS), ctx->d_scalars + kGatherTotalsSlot + u);
    {
      LaunchTimer lt(ctx, pad ? "gather_lengths_scan_kernel<PAD>" : "gather_lengths_scan_kernel");
      launch_compact(ctx, lengths_scan, a.sc, a);
    }
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);
  }
  if (n == 0) return out;
  std::vector<unsigned long long> totals(utf8.size());
  read_scalars(ctx, kGatherTotalsSlot, int(utf8.size()), totals.data());
  for (size_t u = 0; u < utf8.size(); ++u) {
    const Column& src = *in[utf8[u]];
    Column& o = out[utf8[u]];
    FG_CHECK(totals[u] < (1ull << 31), FLOCKGPU_ERR_UNSUPPORTED, "gather: Utf8 result column \"%s\" exceeds 2^31-1 bytes", src.name.c_str());
    o.values_bytes = int64_t(totals[u]);
    o.data = alloc(ctx, size_t(totals[u]));
    if (totals[u] > 0) {
      {
        LaunchTimer lt(ctx, pad ? "gather_utf8_copy_kernel<PAD>" : "gather_utf8_copy_kernel");
        copy<<<stream_grid(ctx, (n + 31) / 32, GA_THREADS / 32), GA_THREADS, 0, ctx->stream>>>(
            static_cast<const uint8_t*>(src.values()), src.offs(), d_idx, o.offsets->as<int32_t>(), o.data->as<uint8_t>(), n);
      }
      FG_CUDA(cudaGetLastError());
      count_launch(ctx);
    }
  }
  return out;
}

TablePtr gather_rows(const CtxPtr& ctx, const Table& in, const std::vector<int>& cols, const uint32_t* d_idx, int64_t n_idx) {
  in.dense();
  auto out = std::make_shared<Table>();
  out->ctx = ctx;
  out->metadata = in.metadata;
  out->num_rows = n_idx;
  std::vector<const Column*> src;
  for (int c : cols) {
    FG_CHECK(c >= 0 && c < int(in.cols.size()), FLOCKGPU_ERR_INVALID, "gather: column %d out of range", c);
    src.push_back(&in.cols[c]);
  }
  out->cols = gather_columns(ctx, src, d_idx, n_idx);
  return out;
}

}  // namespace fg
