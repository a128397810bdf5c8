// hash_join.cu -- K3/K4: HashJoinExec { mode: Partitioned, join_type: Inner | Left | Right | Full | Semi | Anti }.
//
// Reference operator (DataFusion fork, not in tree; used at flock/src/distributed_plan/planner.rs:169,
// :239 and serialised in flock/src/tests/data/plan/join.json): build a hash map over ALL left batches
// (hash -> row indices), then for every right batch emit (left_idx, right_idx) for each pair of equal
// keys and materialise `take(left columns) ++ take(right columns)`.  NULL keys never match (no NULLs on
// this path); duplicate keys on both sides give the full cross product.
//
// GPU design: an open-addressing table with ONE slot per DISTINCT build key -- the slot holds a
// representative build row (key equality is checked against the immutable build columns, so there is no
// publish race), the head of a linked list threading all build rows of that key (`next[row]`), and their
// count.  Heavily duplicated keys (NEXMark q5 joins 6.5 M (auction, num) rows on `num`, ~850 distinct
// values; q3's hot sellers) therefore cost one probe step, not one per duplicate.  The SMALLER input is
// the build side (the reference always builds on the left; which side is hashed is not observable).
//   join_build_kernel        claim / find the key's slot, push the row on its list
//   join_count_scan_kernel   per probe row: number of matches -> exclusive offsets (the grid-wide prefix
//                            protocol of compact.cuh, single pass) and the total pair count
//   join_emit_kernel         second walk (table lines are L2-hot) writes the (build, probe) index pairs
//   join_one_kernel          build side of ONE row (q5 / q7 join with a global aggregate): a stable equality
//                            compaction over the probe side, no table
// and gather.cu materialises the output columns (Utf8 included).  The kernels are instantiated per key shape:
// one 4-byte key, one 8-byte key, or the general form (two packed columns / row comparison for Utf8 keys).
//
// The other join types keep the rule that the smaller input is hashed, so each has a form for its preserved (or
// filtered) side being streamed and one for it being hashed:
//   preserved side streamed   (Left with right hashed, Right with left hashed, Full): the count kernel counts
//                             max(matches, 1) per probe row and the emit kernel writes the pad sentinel JOIN_EMPTY as
//                             the build row of a row without a match -- the same two launches as Inner
//   Semi / Anti, left streamed  join_filter_kernel: one stable compaction of the left rows, a row survives when its key
//                             has a slot (Semi) or has none (Anti); no pairs, no chain walk
//   preserved / filtered side hashed  (Left with left hashed, Right with right hashed, Full, Semi / Anti with left
//                             hashed): visits are recorded PER SLOT -- the build pass stores each build row's slot, a
//                             probe that finds a slot stores visited[slot] = 1 (idempotent, no atomics, no chain walk) --
//                             and join_visited_kernel compacts the build rows whose slot was (Semi) or was not visited,
//                             in build-row order.  Outer types append those rows after the pairs with the sentinel on
//                             the probe side; for Semi / Anti they are the whole output.
// A row with a NULL key has no slot: it matches nothing, is unvisited, and is kept by every type that keeps its side.
#include <algorithm>

#include "compact.cuh"
#include "device_utils.cuh"
#include "internal.h"
#include "rowkeys.cuh"

namespace fg {

constexpr unsigned JOIN_EMPTY = ~0u;

struct JoinSide {
  int64_t n_rows;
  int32_t packed;
  int32_t pad;
  const void* key0;  // the key column when the join has ONE fixed-width key (kernels instantiated with KW = 4 / 8)
  int32_t n_null_cols, pad2;  // key columns that carry validity bytes: a row with a NULL key matches nothing (NULL != NULL)
  const uint8_t* key_valid[MAX_KEY_COLS];
  KeyPack pack;
  RowKeys rk;
  ColRef cols[MAX_IN_COLS];
};

struct JoinTable {
  unsigned* rep;           // [cap] representative build row of the slot's key, JOIN_EMPTY = free
  unsigned* head;          // [cap] most recently pushed build row of that key
  unsigned* cnt;           // [cap] number of build rows with that key
  unsigned* next;          // [build rows] next build row with the same key, JOIN_EMPTY = end
  unsigned long long cap;  // power of two
  struct JoinSlot* slots;  // KW = 4: the table proper (below); rep / head / cnt are unused, `next` holds row + 1
  unsigned* slot_of;       // [build rows] slot of the row's key, JOIN_EMPTY for a NULL key (hashed preserved side only)
  uint8_t* visited;        // [cap] 1 = some probe row found this slot (hashed preserved side only)
};

// One 4-byte key (every NEXMark join but q5's): the KEY LIVES IN THE SLOT.  A probe is one 16-byte load -- key, list
// head and count arrive together -- where the representative-row table needs three dependent reads (rep[slot], the
// build key column at that row, cnt[slot]) in three cache lines; the build claims a slot with one CAS that returns the
// resident key.  ncu on q8 (profiles/r2_join_gather_ncu.md): the representative-row kernels sat at 9-25 % issue
// utilisation with 55-140 warps stalled on those loads per issued instruction.  All-zero = empty, so the table is
// initialised by one memset: `tag_key` carries an occupied bit above the key, `head` and next[] hold row + 1.
struct __align__(16) JoinSlot {
  unsigned long long tag_key;  // 0 = free, else (1 << 63) | key
  unsigned head;               // most recently pushed build row + 1
  unsigned cnt;                // build rows with this key
};
constexpr unsigned long long JOIN_TAG = 1ull << 63;
// Capacity stays a power of two >= 2 x build rows (load 0.3 - 0.5).  A table at load 0.6 of any capacity (slot = high
// half of hash x capacity: 67 MB instead of 134 MB for q8's 2.5 M persons, inside the L2) was measured and is SLOWER
// (run 27: build 59 -> 83 us, count 54 -> 93 us): linear probing at that load makes 2-3 x the dependent accesses, and
// those, not the table's footprint, are what the kernels wait for.
// KW = 4 / 8: one fixed-width key column, read straight from JoinSide::key0 (every NEXMark join); KW = 0: the general
// form (two packed columns, or row comparison for Utf8 / wide keys).  The general form cost ~140 lane-instructions per
// probe row on q5 (dynamic indexing of the column table in parameter space, width and mode branches).
__device__ __forceinline__ bool key_is_null(const JoinSide& s, int64_t row) {
  for (int i = 0; i < s.n_null_cols; ++i)
    if (!s.key_valid[i][row]) return true;
  return false;
}

template <int KW>
__device__ __forceinline__ unsigned long long side_hash(const JoinSide& s, int64_t row, unsigned long long* key) {
  if (KW == 4) {
    *key = static_cast<const uint32_t*>(s.key0)[row];
    return fmix64(*key);
  }
  if (KW == 8) {
    *key = static_cast<const unsigned long long*>(s.key0)[row];
    return fmix64(*key);
  }
  if (s.packed) {
    *key = pack_key(s.pack, s.cols, row);
    return fmix64(*key);
  }
  *key = 0;
  return hash_row(s.rk, s.cols, row);
}

// Does build row `r` carry the key (`key` / row `row` of side `other`)?
template <int KW>
__device__ __forceinline__ bool build_row_matches(const JoinSide& build, unsigned r, const JoinSide& other, int64_t row, unsigned long long key) {
  if (KW == 4) return static_cast<const uint32_t*>(build.key0)[r] == uint32_t(key);
  if (KW == 8) return static_cast<const unsigned long long*>(build.key0)[r] == key;
  return build.packed ? pack_key(build.pack, build.cols, int64_t(r)) == key : rows_equal(build.rk, build.cols, int64_t(r), other.rk, other.cols, row);
}

// REC: also store each build row's slot in t.slot_of (the hashed side is preserved or filtered: join_visited_kernel)
template <int KW, bool REC = false>
__global__ void __launch_bounds__(256) join_build_kernel(const __grid_constant__ JoinSide build, const JoinTable t) {
  for (int64_t row = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; row < build.n_rows; row += int64_t(gridDim.x) * blockDim.x) {
    if (key_is_null(build, row)) {  // never enters the table: nothing can match it
      if (REC) t.slot_of[row] = JOIN_EMPTY;
      continue;
    }
    unsigned long long key;
    unsigned long long slot = side_hash<KW>(build, row, &key) & (t.cap - 1);
    if (KW == 4) {
      const unsigned long long want = JOIN_TAG | key;
      while (true) {
        unsigned long long cur = t.slots[slot].tag_key;
        if (cur == 0ull) cur = atomicCAS(&t.slots[slot].tag_key, 0ull, want);
        if (cur == 0ull || cur == want) break;
        slot = (slot + 1) & (t.cap - 1);
      }
      t.next[row] = atomicExch(&t.slots[slot].head, unsigned(row) + 1u);
      atomicAdd(&t.slots[slot].cnt, 1u);
      if (REC) t.slot_of[row] = unsigned(slot);
      continue;
    }
    while (true) {
      unsigned r = t.rep[slot];
      if (r == JOIN_EMPTY) {
        r = atomicCAS(&t.rep[slot], JOIN_EMPTY, unsigned(row));
        if (r == JOIN_EMPTY) break;  // claimed: this row represents the key
      }
      if (build_row_matches<KW>(build, r, build, row, key)) break;
      slot = (slot + 1) & (t.cap - 1);
    }
    t.next[row] = atomicExch(&t.head[slot], unsigned(row));
    atomicAdd(&t.cnt[slot], 1u);
    if (REC) t.slot_of[row] = unsigned(slot);
  }
}

// Slot of the key of probe row `row`, or ~0 when no build row has it.
// (KW = 4: *head receives the list head (row + 1) and *cnt the number of build rows of the key, from the same load)
template <int KW>
__device__ __forceinline__ unsigned long long find_slot(const JoinSide& build, const JoinSide& probe, const JoinTable& t, int64_t row, unsigned* head,
                                                        unsigned* cnt) {
  if (key_is_null(probe, row)) return ~0ull;
  unsigned long long key;
  unsigned long long slot = side_hash<KW>(probe, row, &key) & (t.cap - 1);
  if (KW == 4) {
    const unsigned long long want = JOIN_TAG | key;
    while (true) {
      const uint4 s = *reinterpret_cast<const uint4*>(&t.slots[slot]);
      const unsigned long long tag = ((unsigned long long)s.y << 32) | s.x;
      if (tag == 0ull) return ~0ull;
      if (tag == want) {
        *head = s.z;
        *cnt = s.w;
        return slot;
      }
      slot = (slot + 1) & (t.cap - 1);
    }
  }
  while (true) {
    const unsigned r = t.rep[slot];
    if (r == JOIN_EMPTY) return ~0ull;
    if (build_row_matches<KW>(build, r, probe, row, key)) return slot;
    slot = (slot + 1) & (t.cap - 1);
  }
}

constexpr int JC_THREADS = 256;
constexpr int JC_ITEMS = 4;
constexpr int JC_TILE = JC_THREADS * JC_ITEMS;

struct JoinCountArgs {
  JoinSide build, probe;
  JoinTable table;
  unsigned* out_off;  // [probe rows + 1] exclusive pair offsets
  CompactScratch sc;  // grid-wide exclusive prefix of the tiles' pair counts (compact.cuh); sc.out_count = total pairs
  unsigned long long* pad_rows;  // JOIN_PAD_PROBE: receives the number of probe rows without a match (zeroed by the host)
};

// Forms of the count / emit kernels beyond Inner's (FORM = 0)
constexpr int JOIN_PAD_PROBE = 1;  // the probe side is preserved: a probe row without a match yields one padded row
constexpr int JOIN_MARK = 2;       // the build side is preserved: record visited[slot]

template <int KW, int FORM = 0>
__global__ void __launch_bounds__(JC_THREADS) join_count_scan_kernel(const __grid_constant__ JoinCountArgs a) {
  __shared__ CompactSmem<1, 16> sm;
  __shared__ unsigned long long s_warp[JC_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n = a.probe.n_rows;
  long long tile;
  for (int it = 0; (tile = cp_next_tile(sm, a.sc, it)) >= 0; ++it) {
    const int64_t i0 = tile * JC_TILE + int64_t(tid) * JC_ITEMS;
    unsigned cnt[JC_ITEMS];
    unsigned long long local = 0;
    unsigned pads = 0;
#pragma unroll
    for (int k = 0; k < JC_ITEMS; ++k) {
      unsigned c = 0;
      if (i0 + k < n) {
        unsigned head = 0, in_slot = 0;
        const unsigned long long slot = find_slot<KW>(a.build, a.probe, a.table, i0 + k, &head, &in_slot);
        if (slot != ~0ull) {
          c = KW == 4 ? in_slot : a.table.cnt[slot];
          if (FORM & JOIN_MARK) a.table.visited[slot] = 1;
        }
        if ((FORM & JOIN_PAD_PROBE) && c == 0) {
          c = 1;
          ++pads;
        }
      }
      cnt[k] = c;
      local += c;
    }
    if (FORM & JOIN_PAD_PROBE) {
      pads = warp_sum(pads);
      if (lane == 0 && pads) atomicAdd(a.pad_rows, (unsigned long long)pads);
    }
    unsigned long long incl = warp_inclusive_sum(local);
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned long long warp_base = 0, tile_total = 0;
#pragma unroll
    for (int w = 0; w < JC_THREADS / 32; ++w) {
      unsigned long long v = s_warp[w];
      if (w < warp) warp_base += v;
      tile_total += v;
    }
    // exclusive prefix over the tiles: the whole CTA looks back (256 predecessors per step) or, when every tile is
    // resident, reads its predecessors' self-validating count words
    if (a.sc.single_wave) cp_grid_prefix(sm, a.sc, tile, tile_total);
    else cp_block_lookback(sm, a.sc, tile, tile_total);
    unsigned long long run = sm.excl + warp_base + (incl - local);
#pragma unroll
    for (int k = 0; k < JC_ITEMS; ++k) {
      if (i0 + k < n) a.out_off[i0 + k] = unsigned(run);
      run += cnt[k];
    }
    if (tile == a.sc.num_tiles - 1 && tid == 0) a.out_off[n] = unsigned(sm.excl + tile_total);
    __syncthreads();  // sm / s_warp are reused by the next tile
  }
}

// ---- build side of ONE row (NEXMark q5 / q7 join a relation with a global aggregate): no table, no chains -- the
// probe is an equality filter.  One stable compaction pass writes the matching probe rows; every pair's build row is 0.
struct JoinOneArgs {
  CompactScratch sc;
  const void* probe_key;
  const void* build_key;  // device pointer to the single build key
  int64_t n_rows;
  unsigned* probe_idx;
};

template <int KW>
__global__ void __launch_bounds__(CP_THREADS) join_one_kernel(const __grid_constant__ JoinOneArgs a) {
  constexpr int E = 4, I = 16, G = I / E;
  constexpr int TILE = CP_THREADS * I;
  __shared__ CompactSmem<E, I> sm;
  const int tid = threadIdx.x, warp = tid >> 5;
  const unsigned long long want = KW == 4 ? (unsigned long long)*static_cast<const uint32_t*>(a.build_key) : *static_cast<const unsigned long long*>(a.build_key);
  long long tile;
  for (int it = 0; (tile = cp_next_tile(sm, a.sc, it)) >= 0; ++it) {
    const int64_t tile_base = tile * TILE;
    unsigned long long bits = 0;
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const int64_t r0 = tile_base + (int64_t(g) * CP_THREADS + tid) * E;
      unsigned nib = 0;
      if (r0 + 3 < a.n_rows) {
        if (KW == 4) {
          const uint4 k = *reinterpret_cast<const uint4*>(static_cast<const uint32_t*>(a.probe_key) + r0);
          nib = unsigned(k.x == uint32_t(want)) | (unsigned(k.y == uint32_t(want)) << 1) | (unsigned(k.z == uint32_t(want)) << 2) | (unsigned(k.w == uint32_t(want)) << 3);
        } else {
          const unsigned long long* p = static_cast<const unsigned long long*>(a.probe_key) + r0;
          const ulonglong2 k01 = *reinterpret_cast<const ulonglong2*>(p), k23 = *reinterpret_cast<const ulonglong2*>(p + 2);
          nib = unsigned(k01.x == want) | (unsigned(k01.y == want) << 1) | (unsigned(k23.x == want) << 2) | (unsigned(k23.y == want) << 3);
        }
      } else {
        for (int e = 0; e < E; ++e) {
          if (r0 + e >= a.n_rows) break;
          const unsigned long long k = KW == 4 ? (unsigned long long)static_cast<const uint32_t*>(a.probe_key)[r0 + e]
                                               : static_cast<const unsigned long long*>(a.probe_key)[r0 + e];
          nib |= unsigned(k == want) << e;
        }
      }
      bits |= (unsigned long long)nib << (g * E);
    }
    unsigned lane_prefix[G];
    cp_rank_tile<E, I>(sm, a.sc, tile, bits, lane_prefix);
    if (bits && sm.tile_total) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const unsigned nib = unsigned(bits >> (g * E)) & 0xfu;
        if (!nib) continue;
        const int64_t r0 = tile_base + (int64_t(g) * CP_THREADS + tid) * E;
        const int64_t pos0 = int64_t(sm.excl) + sm.group_warp[g][warp] + lane_prefix[g];
#pragma unroll
        for (int e = 0; e < E; ++e)
          if ((nib >> e) & 1u) a.probe_idx[pos0 + __popc(nib & ((1u << e) - 1u))] = unsigned(r0 + e);
      }
    }
    __syncthreads();
  }
}

struct JoinEmitArgs {
  JoinSide build, probe;
  JoinTable table;
  const unsigned* off;
  unsigned* build_idx;
  unsigned* probe_idx;
};

template <int KW, int FORM = 0>
__global__ void __launch_bounds__(256) join_emit_kernel(const __grid_constant__ JoinEmitArgs a) {
  for (int64_t row = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; row < a.probe.n_rows; row += int64_t(gridDim.x) * blockDim.x) {
    unsigned pos = a.off[row];
    if (a.off[row + 1] == pos) continue;
    unsigned head = 0, in_slot = 0;
    const unsigned long long slot = find_slot<KW>(a.build, a.probe, a.table, row, &head, &in_slot);
    if ((FORM & JOIN_PAD_PROBE) && slot == ~0ull) {  // no match: one row, build side padded
      a.build_idx[pos] = JOIN_EMPTY;
      a.probe_idx[pos] = unsigned(row);
      continue;
    }
    if (KW == 4) {
      for (unsigned r1 = head; r1 != 0u; r1 = a.table.next[r1 - 1u]) {  // row + 1 links, 0 ends the list
        a.build_idx[pos] = r1 - 1u;
        a.probe_idx[pos] = unsigned(row);
        ++pos;
      }
      continue;
    }
    for (unsigned r = a.table.head[slot]; r != JOIN_EMPTY; r = a.table.next[r]) {
      a.build_idx[pos] = r;
      a.probe_idx[pos] = unsigned(row);
      ++pos;
    }
  }
}

// ---- Semi / Anti with the left side streamed, and the hashed side's (un)visited rows: one stable compaction each, on
// the join_one_kernel skeleton.  Survivors are written in row order, so Semi / Anti keep the left input order.
struct JoinSelectArgs {
  CompactScratch sc;
  JoinSide build, probe;  // join_filter_kernel: probe = the rows compacted
  JoinTable table;
  int64_t n_rows;         // rows compacted
  unsigned* out_idx;
};

template <class Pred>
__device__ __forceinline__ void join_select_rows(const JoinSelectArgs& a, Pred survives) {
  constexpr int E = 4, I = 16, G = I / E;
  constexpr int TILE = CP_THREADS * I;
  __shared__ CompactSmem<E, I> sm;
  const int tid = threadIdx.x;
  long long tile;
  for (int it = 0; (tile = cp_next_tile(sm, a.sc, it)) >= 0; ++it) {
    const int64_t tile_base = tile * TILE;
    unsigned long long bits = 0;
#pragma unroll
    for (int k = 0; k < I; ++k) {
      const int64_t r = tile_base + cp_item_index<E>(k, tid);
      if (r < a.n_rows && survives(r)) bits |= 1ull << k;
    }
    unsigned lane_prefix[G];
    cp_rank_tile<E, I>(sm, a.sc, tile, bits, lane_prefix);
    if (bits && sm.tile_total) {
      unsigned long long m = bits;
      while (m) {
        const int k = __ffsll((long long)m) - 1;
        m &= m - 1;
        a.out_idx[cp_position<E, I>(sm, bits, k, lane_prefix)] = unsigned(tile_base + cp_item_index<E>(k, tid));
      }
    }
    __syncthreads();
  }
}

// left rows (streamed) whose key has a slot in the right side's table (Semi) or has none (Anti; a NULL key has none)
template <int KW, bool ANTI>
__global__ void __launch_bounds__(CP_THREADS) join_filter_kernel(const __grid_constant__ JoinSelectArgs a) {
  join_select_rows(a, [&](int64_t r) {
    unsigned head = 0, in_slot = 0;
    return (find_slot<KW>(a.build, a.probe, a.table, r, &head, &in_slot) != ~0ull) != ANTI;
  });
}

// build rows whose slot some probe row found (VISITED: Semi) or none did (outer types, Anti; a NULL key has no slot)
template <bool VISITED>
__global__ void __launch_bounds__(CP_THREADS) join_visited_kernel(const __grid_constant__ JoinSelectArgs a) {
  join_select_rows(a, [&](int64_t r) {
    const unsigned s = a.table.slot_of[r];
    return (s != JOIN_EMPTY && a.table.visited[s]) == VISITED;
  });
}

// every probe row that finds its key's slot marks it visited (Semi / Anti with the left side hashed: no pairs needed)
template <int KW>
__global__ void __launch_bounds__(256) join_mark_kernel(const __grid_constant__ JoinSide build, const __grid_constant__ JoinSide probe, const JoinTable t) {
  for (int64_t row = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; row < probe.n_rows; row += int64_t(gridDim.x) * blockDim.x) {
    unsigned head = 0, in_slot = 0;
    const unsigned long long slot = find_slot<KW>(build, probe, t, row, &head, &in_slot);
    if (slot != ~0ull) t.visited[slot] = 1;
  }
}

// ------------------------------------------------------------------------------------------------
static void fill_side(const Table& t, const std::vector<int>& keys, bool packed, JoinSide* s) {
  FG_CHECK(t.cols.size() <= size_t(MAX_IN_COLS), FLOCKGPU_ERR_UNSUPPORTED, "hash_join: more than %d columns on one side", MAX_IN_COLS);
  s->n_rows = t.num_rows;
  s->packed = packed ? 1 : 0;
  for (size_t i = 0; i < t.cols.size(); ++i) {
    s->cols[i].data = t.cols[i].values();
    s->cols[i].offsets = t.cols[i].offs();
    s->cols[i].dtype = t.cols[i].dtype;
    s->cols[i].chunk_shift = 0;
    s->cols[i].chunks = nullptr;
    s->cols[i].validity = nullptr;  // key equality between the sides is value equality: rows with NULL keys are skipped up front
  }
  s->rk.n = int(keys.size());
  s->n_null_cols = 0;
  for (size_t i = 0; i < keys.size(); ++i) {
    s->rk.col[i] = keys[i];
    if (t.cols[keys[i]].validity) s->key_valid[s->n_null_cols++] = t.cols[keys[i]].valid();
  }
  if (packed) {
    s->pack.n = int(keys.size());
    for (size_t i = 0; i < keys.size(); ++i) {
      s->pack.col[i] = keys[i];
      s->pack.width[i] = t.cols[keys[i]].width();
    }
  }
}

static int grid_for(const CtxPtr& ctx, int64_t items, int threads, int per_sm) {
  return int(std::max<int64_t>(1, std::min<int64_t>((items + threads - 1) / threads, int64_t(ctx->sm_count) * per_sm)));
}

static TablePtr join_typed(const CtxPtr& ctx, const Table& L, const Table& R, const std::vector<int>& left_keys, const std::vector<int>& right_keys,
                           const std::vector<int>& widths, bool packed, bool null_key, int join_type);

TablePtr hash_join(const CtxPtr& ctx, const TablePtr& left_ptr, const TablePtr& right_ptr, const std::vector<int>& left_keys,
                   const std::vector<int>& right_keys, int join_type) {
  FG_CHECK(join_type >= FLOCKGPU_JOIN_INNER && join_type <= FLOCKGPU_JOIN_ANTI, FLOCKGPU_ERR_INVALID, "hash_join: unknown join type %d", join_type);
  const Table& L = *left_ptr;
  const Table& R = *right_ptr;
  // one side is a single row and the other a group-by result still in table form (NEXMark q5: num = MAX(num)):
  // an equality selection over the table, no rows are materialised for the join (Inner only: the other types take the
  // general path below, which is correct for one-row and deferred inputs as they are)
  if (join_type == FLOCKGPU_JOIN_INNER && left_keys.size() == 1 && right_keys.size() == 1) {
    if (std::shared_ptr<DeferredTable> d = left_ptr->deferred)
      if (TablePtr t = d->select_equal(L, left_keys[0], right_ptr, right_keys[0], true)) return t;
    if (std::shared_ptr<DeferredTable> d = right_ptr->deferred)
      if (TablePtr t = d->select_equal(R, right_keys[0], left_ptr, left_keys[0], false)) return t;
  }
  L.dense();
  R.dense();
  FG_CHECK(!left_keys.empty() && left_keys.size() == right_keys.size(), FLOCKGPU_ERR_INVALID, "hash_join: key lists must be non-empty and of equal length");
  FG_CHECK(left_keys.size() <= size_t(MAX_KEY_COLS), FLOCKGPU_ERR_UNSUPPORTED, "hash_join: more than %d key columns", MAX_KEY_COLS);
  std::vector<int> widths;
  for (size_t i = 0; i < left_keys.size(); ++i) {
    int lk = left_keys[i], rk = right_keys[i];
    FG_CHECK(lk >= 0 && lk < int(L.cols.size()) && rk >= 0 && rk < int(R.cols.size()), FLOCKGPU_ERR_INVALID, "hash_join: key column out of range");
    const Column& lc = L.cols[lk];
    const Column& rc = R.cols[rk];
    FG_CHECK(lc.dtype == rc.dtype, FLOCKGPU_ERR_UNSUPPORTED, "hash_join: key types differ (%s vs %s); DataFusion inserts casts before the join",
             dtype_name(lc.dtype), dtype_name(rc.dtype));
    widths.push_back(lc.width());
  }
  const bool packed = keys_packable(widths.data(), int(widths.size()));

  // a NULL key column (one-row global aggregate over empty input) matches nothing
  bool null_key = false;
  for (size_t i = 0; i < left_keys.size(); ++i) null_key |= L.cols[left_keys[i]].all_null || R.cols[right_keys[i]].all_null;
  if (join_type != FLOCKGPU_JOIN_INNER) return join_typed(ctx, L, R, left_keys, right_keys, widths, packed, null_key, join_type);

  auto out = std::make_shared<Table>();
  out->ctx = ctx;
  out->metadata = L.metadata;

  int64_t n_pairs = 0;
  BufferPtr build_idx, probe_idx;
  // hash the smaller input, stream the larger one through it
  const bool swap_sides = R.num_rows < L.num_rows;
  const Table& B = swap_sides ? R : L;
  const Table& P = swap_sides ? L : R;
  if (L.num_rows > 0 && R.num_rows > 0 && !null_key) {
    JoinSide bs{}, ps{};
    fill_side(B, swap_sides ? right_keys : left_keys, packed, &bs);
    fill_side(P, swap_sides ? left_keys : right_keys, packed, &ps);
    // kernel flavour: one fixed-width key column (4 / 8 bytes) or the general form
    const int kw = (packed && widths.size() == 1) ? widths[0] : 0;
    if (kw) {
      bs.key0 = B.cols[(swap_sides ? right_keys : left_keys)[0]].values();
      ps.key0 = P.cols[(swap_sides ? left_keys : right_keys)[0]].values();
    }
    auto by_width = [&](auto&& f) {
      if (kw == 4) f(std::integral_constant<int, 4>{});
      else if (kw == 8) f(std::integral_constant<int, 8>{});
      else f(std::integral_constant<int, 0>{});
    };
    if (kw && B.num_rows == 1 && bs.n_null_cols == 0 && ps.n_null_cols == 0) {
      // one build row: equality filter over the probe side (see join_one_kernel)
      probe_idx = alloc(ctx, size_t(P.num_rows) * 4);
      JoinOneArgs oa{};
      oa.probe_key = ps.key0;
      oa.build_key = bs.key0;
      oa.n_rows = P.num_rows;
      oa.probe_idx = probe_idx->as<unsigned>();
      const int64_t num_tiles = (P.num_rows + CP_THREADS * 16 - 1) / (CP_THREADS * 16);
      by_width([&](auto w) {
        constexpr int KW = decltype(w)::value == 8 ? 8 : 4;
        auto kernel = join_one_kernel<KW>;
        oa.sc = prepare_compact(ctx, num_tiles, resident_ctas(ctx, reinterpret_cast<const void*>(kernel), CP_THREADS), ctx->d_scalars + 4);
        LaunchTimer lt(ctx, "join_one_kernel");
        launch_compact(ctx, kernel, oa.sc, oa);
      });
      FG_CUDA(cudaGetLastError());
      count_launch(ctx);
      unsigned long long total = 0;
      read_scalars(ctx, 4, 1, &total);
      FG_CHECK(total <= (unsigned long long)P.num_rows, FLOCKGPU_ERR_CUDA, "hash_join: corrupt match count");
      n_pairs = int64_t(total);
      if (n_pairs > 0) {
        build_idx = alloc(ctx, size_t(n_pairs) * 4);
        FG_CUDA(cudaMemsetAsync(build_idx->ptr, 0, size_t(n_pairs) * 4, ctx->stream));
      }
    } else {
    unsigned long long cap = 1024;
    while (cap < 2ull * (unsigned long long)B.num_rows) cap <<= 1;
    JoinTable tab{};
    BufferPtr tbuf;
    if (kw == 4) {
      // 16-byte slots (key, head, count), all-zero = empty, then next[build rows]
      tbuf = alloc(ctx, size_t(cap) * sizeof(JoinSlot) + size_t(B.num_rows) * 4);
      FG_CUDA(cudaMemsetAsync(tbuf->ptr, 0, size_t(cap) * sizeof(JoinSlot), ctx->stream));
      tab.slots = tbuf->as<JoinSlot>();
      tab.next = reinterpret_cast<unsigned*>(tab.slots + cap);
      tab.cap = cap;
    } else {
      // rep | head | cnt in one allocation (cap words each), then next[build rows]
      tbuf = alloc(ctx, size_t(cap) * 12 + size_t(B.num_rows) * 4);
      FG_CUDA(cudaMemsetAsync(tbuf->ptr, 0xff, size_t(cap) * 8, ctx->stream));                                  // rep, head = EMPTY
      FG_CUDA(cudaMemsetAsync(static_cast<char*>(tbuf->ptr) + size_t(cap) * 8, 0, size_t(cap) * 4, ctx->stream));  // cnt = 0
      unsigned* w = tbuf->as<unsigned>();
      tab = JoinTable{w, w + cap, w + 2 * cap, w + 3 * cap, cap, nullptr, nullptr, nullptr};
    }
    {
      LaunchTimer lt(ctx, "join_build_kernel");
      by_width([&](auto w) { join_build_kernel<decltype(w)::value><<<grid_for(ctx, B.num_rows, 256, 8), 256, 0, ctx->stream>>>(bs, tab); });
    }
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);

    BufferPtr off = alloc(ctx, size_t(P.num_rows + 1) * 4);
    JoinCountArgs ca{};
    ca.build = bs;
    ca.probe = ps;
    ca.table = tab;
    ca.out_off = off->as<unsigned>();
    const int64_t num_tiles = (P.num_rows + JC_TILE - 1) / JC_TILE;
    by_width([&](auto w) {
      auto kernel = join_count_scan_kernel<decltype(w)::value>;
      ca.sc = prepare_compact(ctx, num_tiles, resident_ctas(ctx, reinterpret_cast<const void*>(kernel), JC_THREADS), ctx->d_scalars + 4);
      LaunchTimer lt(ctx, "join_count_scan_kernel");
      launch_compact(ctx, kernel, ca.sc, ca);
    });
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);
    unsigned long long total = 0;
    read_scalars(ctx, 4, 1, &total);
    FG_CHECK(total < (1ull << 32) - 1, FLOCKGPU_ERR_UNSUPPORTED, "hash_join: %llu output rows exceed 2^32-2", total);
    n_pairs = int64_t(total);
    if (n_pairs > 0) {
      build_idx = alloc(ctx, size_t(n_pairs) * 4);
      probe_idx = alloc(ctx, size_t(n_pairs) * 4);
      JoinEmitArgs ea{};
      ea.build = bs;
      ea.probe = ps;
      ea.table = tab;
      ea.off = off->as<unsigned>();
      ea.build_idx = build_idx->as<unsigned>();
      ea.probe_idx = probe_idx->as<unsigned>();
      {
        LaunchTimer lt(ctx, "join_emit_kernel");
        by_width([&](auto w) { join_emit_kernel<decltype(w)::value><<<grid_for(ctx, P.num_rows, 256, 8), 256, 0, ctx->stream>>>(ea); });
      }
      FG_CUDA(cudaGetLastError());
      count_launch(ctx);
    }
    }  // general build / probe
  }
  out->num_rows = n_pairs;
  if (n_pairs == 0) {
    TablePtr le = empty_like(ctx, L), re = empty_like(ctx, R);
    for (const Column& c : le->cols) out->cols.push_back(c);
    for (const Column& c : re->cols) out->cols.push_back(c);
    return out;
  }
  // output schema is always left ++ right, whichever side was hashed
  const uint32_t* l_idx = (swap_sides ? probe_idx : build_idx)->as<uint32_t>();
  const uint32_t* r_idx = (swap_sides ? build_idx : probe_idx)->as<uint32_t>();
  std::vector<const Column*> lsrc, rsrc;
  for (const Column& c : L.cols) lsrc.push_back(&c);
  for (const Column& c : R.cols) rsrc.push_back(&c);
  for (Column& c : gather_columns(ctx, lsrc, l_idx, n_pairs)) out->cols.push_back(std::move(c));
  for (Column& c : gather_columns(ctx, rsrc, r_idx, n_pairs)) out->cols.push_back(std::move(c));
  return out;
}


// ---- Left / Right / Full / Semi / Anti ------------------------------------------------------------------------------
static TablePtr join_typed(const CtxPtr& ctx, const Table& L, const Table& R, const std::vector<int>& left_keys, const std::vector<int>& right_keys,
                           const std::vector<int>& widths, bool packed, bool null_key, int join_type) {
  const bool semi_anti = join_type == FLOCKGPU_JOIN_SEMI || join_type == FLOCKGPU_JOIN_ANTI;
  const bool keep_left = join_type == FLOCKGPU_JOIN_LEFT || join_type == FLOCKGPU_JOIN_FULL;   // unmatched left rows are kept
  const bool keep_right = join_type == FLOCKGPU_JOIN_RIGHT || join_type == FLOCKGPU_JOIN_FULL;
  // output: left ++ right (left only for Semi / Anti); the side that can be padded is nullable whatever the data
  auto assemble = [&](std::vector<Column> lcols, std::vector<Column> rcols, int64_t rows) {
    auto out = std::make_shared<Table>();
    out->ctx = ctx;
    out->metadata = L.metadata;
    out->num_rows = rows;
    for (Column& c : lcols) {
      c.nullable |= keep_right;
      out->cols.push_back(std::move(c));
    }
    if (!semi_anti)
      for (Column& c : rcols) {
        c.nullable |= keep_left;
        out->cols.push_back(std::move(c));
      }
    return TablePtr(out);
  };

  if (L.num_rows == 0 || R.num_rows == 0 || null_key) {
    // nothing matches: the preserved side(s) padded, no kernel
    switch (join_type) {
      case FLOCKGPU_JOIN_SEMI: return assemble(empty_like(ctx, L)->cols, {}, 0);
      case FLOCKGPU_JOIN_ANTI: return assemble(L.cols, {}, L.num_rows);
      case FLOCKGPU_JOIN_LEFT: return assemble(L.cols, null_columns(ctx, R, L.num_rows), L.num_rows);
      case FLOCKGPU_JOIN_RIGHT: return assemble(null_columns(ctx, L, R.num_rows), R.cols, R.num_rows);
      default: {
        TablePtr lpart = assemble(L.cols, null_columns(ctx, R, L.num_rows), L.num_rows);
        TablePtr rpart = assemble(null_columns(ctx, L, R.num_rows), R.cols, R.num_rows);
        if (R.num_rows == 0) return lpart;
        if (L.num_rows == 0) return rpart;
        return concat_tables(ctx, {lpart, rpart});
      }
    }
  }

  // hash the smaller input, stream the larger one through it (as Inner)
  const bool swap_sides = R.num_rows < L.num_rows;
  const Table& B = swap_sides ? R : L;
  const Table& P = swap_sides ? L : R;
  // the hashed side needs visit records when its unmatched rows are output (outer) or it is the side Semi / Anti filter
  const bool keep_build = semi_anti ? !swap_sides : (swap_sides ? keep_right : keep_left);
  const bool keep_probe = !semi_anti && (swap_sides ? keep_left : keep_right);
  JoinSide bs{}, ps{};
  fill_side(B, swap_sides ? right_keys : left_keys, packed, &bs);
  fill_side(P, swap_sides ? left_keys : right_keys, packed, &ps);
  const int kw = (packed && widths.size() == 1) ? widths[0] : 0;
  if (kw) {
    bs.key0 = B.cols[(swap_sides ? right_keys : left_keys)[0]].values();
    ps.key0 = P.cols[(swap_sides ? left_keys : right_keys)[0]].values();
  }
  auto by_width = [&](auto&& f) {
    if (kw == 4) f(std::integral_constant<int, 4>{});
    else if (kw == 8) f(std::integral_constant<int, 8>{});
    else f(std::integral_constant<int, 0>{});
  };

  unsigned long long cap = 1024;
  while (cap < 2ull * (unsigned long long)B.num_rows) cap <<= 1;
  FG_CHECK(cap < (1ull << 32), FLOCKGPU_ERR_UNSUPPORTED, "hash_join: %lld build rows exceed the typed join's slot range", (long long)B.num_rows);
  const size_t slots_bytes = kw == 4 ? size_t(cap) * sizeof(JoinSlot) : size_t(cap) * 12;
  const size_t next_bytes = size_t(B.num_rows) * 4;
  const size_t visit_bytes = keep_build ? next_bytes + size_t(cap) : 0;  // slot_of[build rows], visited[cap]
  BufferPtr tbuf = alloc(ctx, slots_bytes + next_bytes + visit_bytes);
  JoinTable tab{};
  if (kw == 4) {
    FG_CUDA(cudaMemsetAsync(tbuf->ptr, 0, slots_bytes, ctx->stream));
    tab.slots = tbuf->as<JoinSlot>();
    tab.next = reinterpret_cast<unsigned*>(tab.slots + cap);
    tab.cap = cap;
  } else {
    FG_CUDA(cudaMemsetAsync(tbuf->ptr, 0xff, size_t(cap) * 8, ctx->stream));
    FG_CUDA(cudaMemsetAsync(static_cast<char*>(tbuf->ptr) + size_t(cap) * 8, 0, size_t(cap) * 4, ctx->stream));
    unsigned* w = tbuf->as<unsigned>();
    tab = JoinTable{w, w + cap, w + 2 * cap, w + 3 * cap, cap, nullptr, nullptr, nullptr};
  }
  if (keep_build) {
    tab.slot_of = reinterpret_cast<unsigned*>(static_cast<char*>(tbuf->ptr) + slots_bytes + next_bytes);
    tab.visited = reinterpret_cast<uint8_t*>(tab.slot_of + B.num_rows);
    FG_CUDA(cudaMemsetAsync(tab.visited, 0, size_t(cap), ctx->stream));
  }
  {
    LaunchTimer lt(ctx, keep_build ? "join_build_kernel<REC>" : "join_build_kernel");
    by_width([&](auto w) {
      constexpr int KW = decltype(w)::value;
      (keep_build ? join_build_kernel<KW, true> : join_build_kernel<KW, false>)<<<grid_for(ctx, B.num_rows, 256, 8), 256, 0, ctx->stream>>>(bs, tab);
    });
  }
  FG_CUDA(cudaGetLastError());
  count_launch(ctx);

  // one stable compaction (join_filter_kernel / join_visited_kernel) of `n` rows into `out_idx`, its count to d_scalars[slot]
  auto select = [&](auto kernel, const char* label, int64_t n, unsigned* out_idx, int slot) {
    JoinSelectArgs sa{};
    sa.build = bs;
    sa.probe = ps;
    sa.table = tab;
    sa.n_rows = n;
    sa.out_idx = out_idx;
    const int64_t num_tiles = (n + CP_THREADS * 16 - 1) / (CP_THREADS * 16);
    sa.sc = prepare_compact(ctx, num_tiles, resident_ctas(ctx, reinterpret_cast<const void*>(kernel), CP_THREADS), ctx->d_scalars + slot);
    {
      LaunchTimer lt(ctx, label);
      launch_compact(ctx, kernel, sa.sc, sa);
    }
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);
  };

  if (semi_anti) {
    // left rows, in left order, through one index vector
    const bool anti = join_type == FLOCKGPU_JOIN_ANTI;
    BufferPtr idx = alloc(ctx, size_t(L.num_rows) * 4);
    if (swap_sides) {
      // left streamed: a row survives on whether its key has a slot
      by_width([&](auto w) {
        constexpr int KW = decltype(w)::value;
        select(anti ? join_filter_kernel<KW, true> : join_filter_kernel<KW, false>, anti ? "join_filter_kernel<ANTI>" : "join_filter_kernel<SEMI>",
               L.num_rows, idx->as<unsigned>(), 4);
      });
    } else {
      // left hashed: the right rows mark the slots they find, then the left rows are selected on their slot's mark
      {
        LaunchTimer lt(ctx, "join_mark_kernel");
        by_width([&](auto w) { join_mark_kernel<decltype(w)::value><<<grid_for(ctx, P.num_rows, 256, 8), 256, 0, ctx->stream>>>(bs, ps, tab); });
      }
      FG_CUDA(cudaGetLastError());
      count_launch(ctx);
      select(anti ? join_visited_kernel<false> : join_visited_kernel<true>, anti ? "join_visited_kernel<UNVISITED>" : "join_visited_kernel<VISITED>",
             L.num_rows, idx->as<unsigned>(), 4);
    }
    unsigned long long total = 0;
    read_scalars(ctx, 4, 1, &total);
    FG_CHECK(total <= (unsigned long long)L.num_rows, FLOCKGPU_ERR_CUDA, "hash_join: corrupt row count");
    if (total == 0) return assemble(empty_like(ctx, L)->cols, {}, 0);
    std::vector<const Column*> lsrc;
    for (const Column& c : L.cols) lsrc.push_back(&c);
    return assemble(gather_columns(ctx, lsrc, idx->as<uint32_t>(), int64_t(total)), {}, int64_t(total));
  }

  // ---- outer: pairs (+ one padded row per unmatched probe row), then the unmatched build rows
  BufferPtr off = alloc(ctx, size_t(P.num_rows + 1) * 4);
  if (keep_probe) FG_CUDA(cudaMemsetAsync(ctx->d_scalars + 6, 0, 8, ctx->stream));
  JoinCountArgs ca{};
  ca.build = bs;
  ca.probe = ps;
  ca.table = tab;
  ca.out_off = off->as<unsigned>();
  ca.pad_rows = ctx->d_scalars + 6;
  const int64_t num_tiles = (P.num_rows + JC_TILE - 1) / JC_TILE;
  auto count_form = [&](auto w, auto form) {
    auto kernel = join_count_scan_kernel<decltype(w)::value, decltype(form)::value>;
    ca.sc = prepare_compact(ctx, num_tiles, resident_ctas(ctx, reinterpret_cast<const void*>(kernel), JC_THREADS), ctx->d_scalars + 4);
    LaunchTimer lt(ctx, keep_probe ? (keep_build ? "join_count_scan_kernel<PAD,MARK>" : "join_count_scan_kernel<PAD>") : "join_count_scan_kernel<MARK>");
    launch_compact(ctx, kernel, ca.sc, ca);
  };
  by_width([&](auto w) {
    if (keep_probe && keep_build) count_form(w, std::integral_constant<int, JOIN_PAD_PROBE | JOIN_MARK>{});
    else if (keep_probe) count_form(w, std::integral_constant<int, JOIN_PAD_PROBE>{});
    else count_form(w, std::integral_constant<int, JOIN_MARK>{});
  });
  FG_CUDA(cudaGetLastError());
  count_launch(ctx);
  BufferPtr unvisited;
  if (keep_build) {
    unvisited = alloc(ctx, size_t(B.num_rows) * 4);
    select(join_visited_kernel<false>, "join_visited_kernel<UNVISITED>", B.num_rows, unvisited->as<unsigned>(), 5);
  }
  unsigned long long sc3[3] = {0, 0, 0};  // pairs incl. padded probe rows, unmatched build rows, padded probe rows
  read_scalars(ctx, 4, 3, sc3);
  const unsigned long long n_unvisited = keep_build ? sc3[1] : 0, n_pad_probe = keep_probe ? sc3[2] : 0;
  FG_CHECK(n_unvisited <= (unsigned long long)B.num_rows && n_pad_probe <= (unsigned long long)P.num_rows, FLOCKGPU_ERR_CUDA, "hash_join: corrupt row count");
  FG_CHECK(sc3[0] + n_unvisited < (1ull << 32) - 1, FLOCKGPU_ERR_UNSUPPORTED, "hash_join: %llu output rows exceed 2^32-2", sc3[0] + n_unvisited);
  const int64_t n_pairs = int64_t(sc3[0]), n_rows = n_pairs + int64_t(n_unvisited);
  BufferPtr build_idx = alloc(ctx, size_t(n_rows) * 4), probe_idx = alloc(ctx, size_t(n_rows) * 4);
  if (n_pairs > 0) {
    JoinEmitArgs ea{};
    ea.build = bs;
    ea.probe = ps;
    ea.table = tab;
    ea.off = off->as<unsigned>();
    ea.build_idx = build_idx->as<unsigned>();
    ea.probe_idx = probe_idx->as<unsigned>();
    {
      LaunchTimer lt(ctx, keep_probe ? "join_emit_kernel<PAD>" : "join_emit_kernel");
      by_width([&](auto w) {
        constexpr int KW = decltype(w)::value;
        (keep_probe ? join_emit_kernel<KW, JOIN_PAD_PROBE> : join_emit_kernel<KW, 0>)<<<grid_for(ctx, P.num_rows, 256, 8), 256, 0, ctx->stream>>>(ea);
      });
    }
    FG_CUDA(cudaGetLastError());
    count_launch(ctx);
  }
  if (n_unvisited > 0) {
    FG_CUDA(cudaMemcpyAsync(build_idx->as<unsigned>() + n_pairs, unvisited->ptr, size_t(n_unvisited) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    FG_CUDA(cudaMemsetAsync(probe_idx->as<unsigned>() + n_pairs, 0xff, size_t(n_unvisited) * 4, ctx->stream));  // JOIN_EMPTY
  }
  // sentinels in build_idx: the padded probe rows; in probe_idx: the unmatched build rows
  const uint32_t* l_idx = (swap_sides ? probe_idx : build_idx)->as<uint32_t>();
  const uint32_t* r_idx = (swap_sides ? build_idx : probe_idx)->as<uint32_t>();
  const bool l_pad = (swap_sides ? n_unvisited : n_pad_probe) > 0, r_pad = (swap_sides ? n_pad_probe : n_unvisited) > 0;
  std::vector<const Column*> lsrc, rsrc;
  for (const Column& c : L.cols) lsrc.push_back(&c);
  for (const Column& c : R.cols) rsrc.push_back(&c);
  std::vector<Column> lcols = gather_columns(ctx, lsrc, l_idx, n_rows, l_pad);
  std::vector<Column> rcols = gather_columns(ctx, rsrc, r_idx, n_rows, r_pad);
  return assemble(std::move(lcols), std::move(rcols), n_rows);
}

}  // namespace fg

using namespace fg;

extern "C" int flockgpu_hash_join(flockgpu_ctx* ctx, const flockgpu_table* left, const flockgpu_table* right, const int32_t* left_keys,
                                  const int32_t* right_keys, int32_t n_keys, flockgpu_table** out) {
  return guarded([&] {
    auto c = core_of(ctx);
    FG_CHECK(out && left && left->table && right && right->table && left_keys && right_keys && n_keys > 0, FLOCKGPU_ERR_INVALID,
             "hash_join: null or empty argument");
    std::lock_guard<std::recursive_mutex> g(c->mu);
    FG_CUDA(cudaSetDevice(c->device));
    std::vector<int> lk(left_keys, left_keys + n_keys), rk(right_keys, right_keys + n_keys);
    *out = wrap_table(hash_join(c, left->table, right->table, lk, rk));
  });
}

extern "C" int flockgpu_hash_join_typed(flockgpu_ctx* ctx, const flockgpu_table* left, const flockgpu_table* right, const int32_t* left_keys,
                                        const int32_t* right_keys, int32_t n_keys, int32_t join_type, flockgpu_table** out) {
  return guarded([&] {
    auto c = core_of(ctx);
    FG_CHECK(out && left && left->table && right && right->table && left_keys && right_keys && n_keys > 0, FLOCKGPU_ERR_INVALID,
             "hash_join: null or empty argument");
    FG_CHECK(join_type >= FLOCKGPU_JOIN_INNER && join_type <= FLOCKGPU_JOIN_ANTI, FLOCKGPU_ERR_INVALID, "hash_join: unknown join type %d", join_type);
    std::lock_guard<std::recursive_mutex> g(c->mu);
    FG_CUDA(cudaSetDevice(c->device));
    std::vector<int> lk(left_keys, left_keys + n_keys), rk(right_keys, right_keys + n_keys);
    *out = wrap_table(hash_join(c, left->table, right->table, lk, rk, join_type));
  });
}
