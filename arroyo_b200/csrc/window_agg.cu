// Tumbling / sliding window keyed aggregate on sm_100a.
//
// Replaces, behind the ArrowOperator surface:
//   TumblingAggregatingWindowFunc  arroyo-worker/src/arrow/tumbling_aggregating_window.rs:250-392
//   SlidingAggregatingWindowFunc   arroyo-worker/src/arrow/sliding_aggregating_window.rs:102-210, :598-737
// and the DataFusion / arrow-rs work they call per batch (SURVEY.md 2b K1-K5, K7):
//   K1 date_bin  K2 sort_to_indices+take+partition  K3 AggregateExec(Partial)
//   K4 AggregateExec(Final)  K5 final projection (window struct, _timestamp)  K7 late-row filter
//
// Design (see DESIGN.md):
//   * one persistent key dictionary per operator (bdict.cuh): buckets of <= 1280 keys, open addressing inside the
//     bucket, dense id = bucket * 1280 + index: a bucket's keys own a contiguous id range.  Keys recur in every
//     pane, so after warm-up a row costs one read-only lookup.
//   * one accumulator block per pane: dense SoA arrays indexed by id (rows, then one 64-bit
//     accumulator per SUM / AVG / MIN / MAX).  Nothing is sorted, gathered or materialised per batch.
//   * ingest, large launches of COUNT / SUM / AVG plans (ingest_two_pass.cuh): rows are radix-partitioned by
//     dictionary bucket (part_kernel), then each bucket is aggregated in shared memory against a lookup table of
//     its keys, fed by per-warp TMA rings, and flushed to its contiguous id range of the pane (agg_kernel).
//     Everything else (small launches, MIN / MAX / f64, partial-row inputs, hot-key streams, rows the two passes
//     hand back): ingest_kernel, one pass -- date_bin (one mulhi) + late test + lookup + one RED per accumulator.
//   * panes live in a ring indexed by (ts / slide) & (R - 1); the device table pane_bins[] says
//     which bin a slot holds.  Rows whose pane is not resident (far future / before the ring) or
//     whose key cannot get an id (dictionary full) are copied to a deferred buffer; the host grows
//     the ring / dictionary at the next sync point and re-ingests them.  No row is lost.
//   * emission merges the panes of a window element-wise over the dense id space, finalises
//     (AVG = sum / count), compacts ids with rows > 0 and writes the output columns including
//     window.start / window.end / _timestamp.  Invertible aggregates (COUNT/SUM/AVG) keep a running
//     window block W += entering pane, W -= leaving pane instead of re-merging width/slide panes.
#include <algorithm>
#include <climits>
#include <deque>
#include <map>
#include <memory>
#include <set>

#include "bdict.cuh"
#include "op.h"
#include "planner.h"

namespace ab {
namespace {

constexpr int MAX_VALS = 4;
constexpr int MAX_ACC = ARROYO_B200_MAX_AGGS + 1;
constexpr int MAX_SEGS = 512;
constexpr int MAX_RING = 4096;
constexpr int RING_INLINE = 64;
constexpr int MAX_MERGE = 4096;
constexpr long long FREE_BIN = LLONG_MIN;

constexpr int THREADS = 256;
constexpr int PAIRS = 2;
constexpr int TILE = THREADS * PAIRS * 2;  // rows per tile

enum AccKind : int { ACC_ROWS = 0, ACC_SUM_I64 = 1, ACC_SUM_F64 = 2, ACC_MIN_I64 = 3, ACC_MAX_I64 = 4 };

struct Counters {
  unsigned long long late_rows;
  unsigned long long deferred;
  unsigned long long lost;
  unsigned long long neg_ts;  // rows with _timestamp < 0 (pre-epoch): the reference panics on them
  unsigned long long max_q;  // newest on-time pane number (ts / slide) seen
  unsigned long long big_vals;  // rows deferred because a value exceeded the exact-AVG guard
  unsigned int n_keys;     // keys in the dictionary (BDict::n_total)
  unsigned int dict_full;  // rows deferred because their bucket was out of ids: the host grows the dictionary
  unsigned long long part_overflow;  // two-pass ingest: rows that did not fit their partition region (skew)
};

struct Segment {
  const long long* key;
  const long long* ts;
  const long long* val[MAX_VALS];
  long long n;
  long long tile_start;
  int vec_ok;
  int pad;
};

struct IngestParams {
  const Segment* segs;
  int n_segs;
  int keyed;
  long long n_tiles;
  BDict dict;
  FastDivU64 slide_div;
  long long slide;
  long long late_bin;
  unsigned long long late_q;  // late_bin / slide (0 when there is no watermark yet)
  unsigned int guard_vals;    // bit x set: value slot x must satisfy |v| < 2^31 (exact-sum AVG, see avg_exact_)
  int combine;                // warp-combine equal (pane, id) before the REDs
  int rows_slot;              // value slot carrying the row count of a partial-aggregate input row, or -1
  int pad2;
  uint32_t ring_mask;
  int n_acc;
  const long long* pane_bins;
  unsigned long long* const* pane_ptrs;
  unsigned long long id_cap;
  // rings of up to RING_INLINE slots travel in the kernel parameters (constant bank): no table upload
  int ring_inline;
  int pad1;
  long long ring_bins[RING_INLINE];
  unsigned long long* ring_ptrs[RING_INLINE];
  int acc_kind[MAX_ACC];
  int acc_val[MAX_ACC];
  Counters* counters;
  unsigned long long* slot_rows;  // on-time rows per ring slot, added by this launch
  long long* d_key;
  long long* d_ts;
  long long* d_val[MAX_VALS];
  unsigned long long defer_cap;
};

// -------------------------------------------------------------------------------------------
// pane blocks
// -------------------------------------------------------------------------------------------
struct InitParams {
  unsigned long long* pane;
  unsigned long long id_cap;
  unsigned long long n;  // ids [0, n) to reset
  int n_acc;
  int acc_kind[MAX_ACC];
};

__global__ void pane_init_kernel(const __grid_constant__ InitParams p) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (; i < p.n; i += stride) {
    for (int a = 0; a < p.n_acc; ++a) {
      unsigned long long v = 0;
      if (p.acc_kind[a] == ACC_MIN_I64) v = (unsigned long long)LLONG_MAX;
      if (p.acc_kind[a] == ACC_MAX_I64) v = (unsigned long long)LLONG_MIN;
      p.pane[a * p.id_cap + i] = v;
    }
  }
}

__device__ __forceinline__ const long long* ldg_ptr(const long long* const* pp) {
  return reinterpret_cast<const long long*>(__ldg(reinterpret_cast<const unsigned long long*>(pp)));
}

// -------------------------------------------------------------------------------------------
// ingest: window-assign + keyed partial aggregate
// -------------------------------------------------------------------------------------------
// RED (fire-and-forget reduction, no return trip).  The pane pointers come out of memory, so the
// compiler only knows them as generic addresses and would emit the slower generic ATOM: state the
// address space explicitly.
__device__ __forceinline__ void red_add_u64(unsigned long long* a, unsigned long long v) {
  asm volatile("red.global.add.u64 [%0], %1;" ::"l"(__cvta_generic_to_global(a)), "l"(v) : "memory");
}
__device__ __forceinline__ void red_add_f64(unsigned long long* a, double v) {
  asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(a)), "d"(v) : "memory");
}
__device__ __forceinline__ void red_min_s64(unsigned long long* a, long long v) {
  asm volatile("red.global.min.s64 [%0], %1;" ::"l"(__cvta_generic_to_global(a)), "l"(v) : "memory");
}
__device__ __forceinline__ void red_max_s64(unsigned long long* a, long long v) {
  asm volatile("red.global.max.s64 [%0], %1;" ::"l"(__cvta_generic_to_global(a)), "l"(v) : "memory");
}

__device__ __forceinline__ long long ring_bin(const IngestParams& p, uint32_t slot) {
  return p.ring_inline ? p.ring_bins[slot] : __ldg(p.pane_bins + slot);
}
__device__ __forceinline__ unsigned long long* ring_ptr(const IngestParams& p, uint32_t slot) {
  return p.ring_inline ? p.ring_ptrs[slot]
                       : reinterpret_cast<unsigned long long*>(__ldg(reinterpret_cast<const unsigned long long*>(p.pane_ptrs + slot)));
}

// Rows travel through the kernel as scalars (key, ts, up to MAX_VALS values): nothing in the hot loop
// is addressable, so nothing is forced into local memory.
struct Vals {
  long long v0, v1, v2, v3;
};
template <int NV>
__device__ __forceinline__ Vals pack_vals(const long long (&v)[NV > 0 ? NV : 1]) {
  Vals o{0, 0, 0, 0};
  if (NV > 0) o.v0 = v[0];
  if (NV > 1) o.v1 = v[NV > 1 ? 1 : 0];
  if (NV > 2) o.v2 = v[NV > 2 ? 2 : 0];
  if (NV > 3) o.v3 = v[NV > 3 ? 3 : 0];
  return o;
}

__device__ __noinline__ void defer_row(const IngestParams& p, long long key, long long ts, long long v0, long long v1,
                                       long long v2, long long v3) {
  unsigned long long idx = atomicAdd(&p.counters->deferred, 1ull);
  if (idx < p.defer_cap) {
    p.d_key[idx] = key;
    p.d_ts[idx] = ts;
    if (p.d_val[0]) p.d_val[0][idx] = v0;
    if (p.d_val[1]) p.d_val[1][idx] = v1;
    if (p.d_val[2]) p.d_val[2][idx] = v2;
    if (p.d_val[3]) p.d_val[3][idx] = v3;
  } else {
    atomicAdd(&p.counters->lost, 1ull);
  }
}

// Accumulator signature: the kinds of accumulators 1..3 packed 3 bits each (0 = none); GENERIC_SIG =
// read kinds / value slots from the params at run time.  The common signatures are compiled as
// straight-line code.
constexpr int GENERIC_SIG = -1;
constexpr int sig_of(int k1, int k2 = 0, int k3 = 0) { return k1 | (k2 << 3) | (k3 << 6); }

__device__ __forceinline__ void red_kind(int kind, unsigned long long* dst, long long v) {
  switch (kind) {
    case ACC_SUM_I64: red_add_u64(dst, (unsigned long long)v); break;
    case ACC_SUM_F64: red_add_f64(dst, (double)v); break;
    case ACC_MIN_I64: red_min_s64(dst, v); break;
    case ACC_MAX_I64: red_max_s64(dst, v); break;
    default: break;
  }
}

// How many original rows an input row stands for: 1, or the carried count of a partial-aggregate row.
__device__ __forceinline__ unsigned long long rows_of(const IngestParams& p, const Vals& v) {
  const int x = p.rows_slot;
  if (x < 0) return 1ull;
  return (unsigned long long)(x == 0 ? v.v0 : x == 1 ? v.v1 : x == 2 ? v.v2 : v.v3);
}

// The RED updates of one row into pane block `pane` (K3: partial aggregate).
template <int NV, int SIG>
__device__ __forceinline__ void accumulate(const IngestParams& p, const Vals& v, unsigned long long* pane, uint32_t id) {
  red_add_u64(pane + id, rows_of(p, v));
  if (SIG == GENERIC_SIG) {
#pragma unroll
    for (int a = 1; a < MAX_ACC; ++a) {
      if (a < p.n_acc) {
        const int x = p.acc_val[a];
        const long long val = x == 0 ? v.v0 : x == 1 ? v.v1 : x == 2 ? v.v2 : v.v3;
        red_kind(p.acc_kind[a], pane + (unsigned long long)a * p.id_cap + id, val);
      }
    }
  } else {
    // at most one value column: every accumulator reads v0
    constexpr int k1 = SIG & 7, k2 = (SIG >> 3) & 7, k3 = (SIG >> 6) & 7;
    if (k1) red_kind(k1, pane + p.id_cap + id, v.v0);
    if (k2) red_kind(k2, pane + 2 * p.id_cap + id, v.v0);
    if (k3) red_kind(k3, pane + 3 * p.id_cap + id, v.v0);
  }
}

__device__ __forceinline__ bool big_one(long long v) { return (unsigned long long)(v + (1ll << 31)) >= (1ull << 32); }
__device__ __forceinline__ bool big_value(unsigned int mask, const Vals& v) {
  return ((mask & 1u) && big_one(v.v0)) || ((mask & 2u) && big_one(v.v1)) || ((mask & 4u) && big_one(v.v2)) ||
         ((mask & 8u) && big_one(v.v3));
}

// Row whose pane is not the thread's cached one (pane boundary inside a warp, tail tiles, tiny
// batches, non-resident pane): look the ring up directly and count the row with its own atomic.
template <int NV, int SIG>
__device__ __noinline__ void slow_row(const IngestParams& p, long long key, long long ts, uint64_t q, long long v0,
                                      long long v1, long long v2, long long v3) {
  const uint32_t slot = (uint32_t)q & p.ring_mask;
  uint32_t id = 0;
  bool ok = ring_bin(p, slot) == (long long)(q * (uint64_t)p.slide);
  if (ok && p.keyed) {
    const uint64_t h = bd_hash(key);
    const ulonglong2* hp = reinterpret_cast<const ulonglong2*>(bd_home(p.dict, key, h));
    const ulonglong2 raw = __ldcg(hp), raw1 = __ldcg(hp + 1);
    id = bd_resolve(p.dict, key, h, raw.x, (uint32_t)raw.y, raw1.x, (uint32_t)raw1.y);
    ok = id < ID_OVERFLOW;
    if (!ok) atomicAdd(&p.counters->dict_full, 1u);
  }
  const Vals v{v0, v1, v2, v3};
  if (ok && NV > 0 && p.guard_vals && big_value(p.guard_vals, v)) {
    atomicAdd(&p.counters->big_vals, 1ull);
    ok = false;
  }
  if (!ok) {
    defer_row(p, key, ts, v0, v1, v2, v3);
    return;
  }
  unsigned long long* pane = ring_ptr(p, slot);
  atomicAdd(p.slot_rows + slot, 1ull);
  accumulate<NV, SIG>(p, v, pane, id);
}

// Per-thread view of the pane ring: the pane (quotient ts / slide) of the previous row lives in
// registers, so the common case -- a warp's rows all in one pane -- touches neither the ring tables nor
// any shared counter.
struct PaneCache {
  uint64_t q = ~0ull;                  // cached pane number
  unsigned long long* ptr = nullptr;   // its block, or nullptr when the pane is not resident
  uint32_t cnt = 0;                    // on-time rows this thread aggregated into it
};

// Warp-combined publication of the per-thread on-time row counts (all 32 lanes must call).
__device__ __forceinline__ void flush_counts(const IngestParams& p, PaneCache& pc, int lane) {
  const unsigned int peers = __match_any_sync(0xffffffffu, pc.q);
  const unsigned int total = __reduce_add_sync(peers, pc.cnt);
  if (total && (__ffs(peers) - 1) == lane)
    atomicAdd(p.slot_rows + ((uint32_t)pc.q & p.ring_mask), (unsigned long long)total);
  pc.cnt = 0;
}

// Divergent half of a hot-path row: residency test, dictionary id, exact-AVG guard.  Returns the id to
// accumulate into, or ID_OVERFLOW when the row was handled out of line (slow path / deferred).
template <int NV, int SIG>
__device__ __forceinline__ uint32_t hot_resolve(const IngestParams& p, const PaneCache& pc, uint64_t& maxq, bool keyed,
                                                long long key, long long ts, uint64_t q, const Vals& v, uint64_t h,
                                                unsigned long long k0, uint32_t id0, unsigned long long k1, uint32_t id1) {
  uint32_t id = ID_OVERFLOW;
  if (q == pc.q && pc.ptr != nullptr) id = keyed ? bd_resolve(p.dict, key, h, k0, id0, k1, id1) : 0u;
  if (NV > 0 && p.guard_vals && big_value(p.guard_vals, v)) {
    // AVG is being derived from the exact integer sum: a value this large could overflow it.  Park the
    // row; the host promotes the operator to f64 AVG accumulators and re-ingests it.
    atomicAdd(&p.counters->big_vals, 1ull);
    defer_row(p, key, ts, v.v0, v.v1, v.v2, v.v3);
    return ID_OVERFLOW;
  }
  if (id >= ID_OVERFLOW) {
    maxq = max(maxq, q);
    slow_row<NV, SIG>(p, key, ts, q, v.v0, v.v1, v.v2, v.v3);
  }
  return id;
}

__device__ __forceinline__ long long shfl_ll(unsigned mask, long long v, int src) {
  return (long long)__shfl_sync(mask, (unsigned long long)v, src);
}

// Combines one accumulator across the lanes of `peers` (same pane, same id); valid in the leader.
__device__ __forceinline__ long long group_reduce(int kind, unsigned peers, long long v) {
  long long r = v;
  bool first = true;
  for (unsigned m = peers; m; m &= m - 1) {
    const long long x = shfl_ll(peers, v, __ffs(m) - 1);
    if (first) {
      r = x;
      first = false;
      continue;
    }
    switch (kind) {
      case ACC_SUM_I64: r = (long long)((unsigned long long)r + (unsigned long long)x); break;
      case ACC_SUM_F64: r = __double_as_longlong(__longlong_as_double(r) + __longlong_as_double(x)); break;
      case ACC_MIN_I64: r = min(r, x); break;
      case ACC_MAX_I64: r = max(r, x); break;
      default: break;
    }
  }
  return r;
}

__device__ __forceinline__ void red_kind_combined(int kind, unsigned long long* dst, long long v) {
  // v is already in the accumulator's domain (f64 bits for ACC_SUM_F64)
  if (kind == ACC_SUM_F64) red_add_f64(dst, __longlong_as_double(v));
  else red_kind(kind, dst, v);
}

// Convergent half: RED updates, after combining lanes of the warp that hit the same (pane, id).  Skewed
// keys (Nexmark: 75 % of the bids on the hot bidder) would otherwise serialise tens of millions of REDs on
// one L2 address; unkeyed aggregates hit a single address by construction.  The neighbour test keeps the
// common case (all ids distinct) at two shuffles and a vote.
template <int NV, int SIG>
__device__ __forceinline__ void combine_accumulate(const IngestParams& p, const PaneCache& pc, bool fast, uint32_t id,
                                                   const Vals& v, int lane) {
  const unsigned long long gkey = fast ? ((unsigned long long)id | (pc.q << 32)) : (0xFFFFFFFF00000000ull | (unsigned)lane);
  const unsigned long long nb = __shfl_xor_sync(0xffffffffu, gkey, 1);
  if (!__any_sync(0xffffffffu, fast && nb == gkey)) {
    if (fast) accumulate<NV, SIG>(p, v, pc.ptr, id);
    return;
  }
  const unsigned peers = __match_any_sync(0xffffffffu, gkey);
  const bool leader = (__ffs(peers) - 1) == lane;
  unsigned long long* pane = pc.ptr;
  if (p.rows_slot < 0) {
    if (fast && leader) red_add_u64(pane + id, (unsigned long long)__popc(peers));
  } else {
    const long long r = group_reduce(ACC_SUM_I64, peers, (long long)rows_of(p, v));
    if (fast && leader) red_add_u64(pane + id, (unsigned long long)r);
  }
  if (SIG == GENERIC_SIG) {
#pragma unroll
    for (int a = 1; a < MAX_ACC; ++a) {
      if (a < p.n_acc) {
        const int x = p.acc_val[a];
        long long val = x == 0 ? v.v0 : x == 1 ? v.v1 : x == 2 ? v.v2 : v.v3;
        const int kind = p.acc_kind[a];
        if (kind == ACC_SUM_F64) val = __double_as_longlong((double)val);
        const long long r = group_reduce(kind, peers, val);
        if (fast && leader) red_kind_combined(kind, pane + (unsigned long long)a * p.id_cap + id, r);
      }
    }
  } else {
    constexpr int k1 = SIG & 7, k2 = (SIG >> 3) & 7, k3 = (SIG >> 6) & 7;
    if (k1) {
      const long long r = group_reduce(k1, peers, k1 == ACC_SUM_F64 ? __double_as_longlong((double)v.v0) : v.v0);
      if (fast && leader) red_kind_combined(k1, pane + p.id_cap + id, r);
    }
    if (k2) {
      const long long r = group_reduce(k2, peers, k2 == ACC_SUM_F64 ? __double_as_longlong((double)v.v0) : v.v0);
      if (fast && leader) red_kind_combined(k2, pane + 2 * p.id_cap + id, r);
    }
    if (k3) {
      const long long r = group_reduce(k3, peers, k3 == ACC_SUM_F64 ? __double_as_longlong((double)v.v0) : v.v0);
      if (fast && leader) red_kind_combined(k3, pane + 3 * p.id_cap + id, r);
    }
  }
}

#ifndef AB_INGEST_PREFETCH
#define AB_INGEST_PREFETCH 1
#endif
#ifndef AB_INGEST_MIN_BLOCKS
#define AB_INGEST_MIN_BLOCKS 4
#endif
template <int NV, int SIG>
__global__ void __launch_bounds__(THREADS, AB_INGEST_MIN_BLOCKS) ingest_kernel(const __grid_constant__ IngestParams p) {
  __shared__ unsigned long long s_late, s_maxq;
  __shared__ unsigned int s_done;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  if (tid == 0) {
    s_late = 0;
    s_maxq = 0;
    s_done = 0;
  }
  __syncthreads();  // the only block barrier: all warps arrive together at kernel start

  PaneCache pc;
  uint32_t late = 0;
  uint64_t maxq = 0;  // newest on-time pane seen (0 = none: pane 0 is 1970)
  const FastDivU64 sd = p.slide_div;
  const bool keyed = p.keyed != 0;

  for (long long tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    int lo = 0, hi = p.n_segs - 1;
    while (lo < hi) {
      int mid = (lo + hi + 1) >> 1;
      if (__ldg(&p.segs[mid].tile_start) <= tile) lo = mid; else hi = mid - 1;
    }
    const Segment* sg = p.segs + lo;
    const long long base = (tile - __ldg(&sg->tile_start)) * TILE;
    const long long nrem = __ldg(&sg->n) - base;
    const int cnt = nrem < TILE ? (int)nrem : TILE;

    // One row per lane per iteration: a warp instruction covers 256 contiguous bytes per column, and
    // with several resident blocks per SM there are well over a thousand independent probe chains in
    // flight per SM (profiles/r01_probe2.txt: occupancy beats rows-per-thread for the scattered part).
    // The next row's columns are requested before the current row is processed, so the streaming loads
    // overlap the dependent probe -> RED chain.  The trip count is uniform so that the warp votes below
    // stay convergent in tail tiles.
    long long nkey = 0, nts = 0;
    long long nv[NV > 0 ? NV : 1] = {0};
    if (tid < cnt) {
      if (keyed) nkey = __ldcs(ldg_ptr(&sg->key) + base + tid);
      nts = __ldcs(ldg_ptr(&sg->ts) + base + tid);
#pragma unroll
      for (int x = 0; x < NV; ++x) nv[x] = __ldcs(ldg_ptr(&sg->val[x]) + base + tid);
    }
#pragma unroll 1
    for (int i = tid; i < TILE; i += THREADS) {
      const bool valid = i < cnt;
      const long long key = nkey, ts = nts;
      long long v[NV > 0 ? NV : 1];
#pragma unroll
      for (int x = 0; x < (NV > 0 ? NV : 1); ++x) v[x] = nv[x];
      ulonglong2 raw = {0, 0}, raw1 = {0, 0};
      const uint64_t h = keyed ? bd_hash(key) : 0ull;
      if (valid && keyed) {
        const ulonglong2* hp = reinterpret_cast<const ulonglong2*>(bd_home(p.dict, key, h));
        raw = __ldcg(hp);
        raw1 = __ldcg(hp + 1);
      }
#if AB_INGEST_PREFETCH
      if (i + THREADS < cnt) {
        if (keyed) nkey = __ldcs(ldg_ptr(&sg->key) + base + i + THREADS);
        nts = __ldcs(ldg_ptr(&sg->ts) + base + i + THREADS);
#pragma unroll
        for (int x = 0; x < NV; ++x) nv[x] = __ldcs(ldg_ptr(&sg->val[x]) + base + i + THREADS);
      }
#endif
      // K1: pane = ts / slide, i.e. bin = ts - ts % slide (tumbling_aggregating_window.rs:65-73)
      const uint64_t q = sd.div((uint64_t)ts);
      // pre-epoch timestamps have no pane (the division is unsigned): reported, never aggregated
      if (valid && ts < 0) atomicAdd(&p.counters->neg_ts, 1ull);
      // K7: late bins are dropped (tumbling :282-291, sliding :631-633)
      const bool live = valid && ts >= 0 && q >= p.late_q;
      late += (valid && !live) ? 1u : 0u;
      // refresh the cached pane when this lane moved to another pane; the vote keeps the warp-combined
      // count flush convergent
      if (__any_sync(0xffffffffu, live && q != pc.q)) {
        flush_counts(p, pc, lane);
        if (live) {
          const uint32_t slot = (uint32_t)q & p.ring_mask;
          const bool resident = ring_bin(p, slot) == (long long)(q * (uint64_t)p.slide);
          pc.q = q;
          pc.ptr = resident ? ring_ptr(p, slot) : nullptr;
          maxq = max(maxq, q);
        }
      }
      const Vals pv = pack_vals<NV>(v);
      uint32_t id = ID_OVERFLOW;
      if (live) id = hot_resolve<NV, SIG>(p, pc, maxq, keyed, key, ts, q, pv, h, raw.x, (uint32_t)raw.y, raw1.x, (uint32_t)raw1.y);
      const bool fast = id < ID_OVERFLOW;
      if (fast) ++pc.cnt;
      if (p.combine) combine_accumulate<NV, SIG>(p, pc, fast, id, pv, lane);
      else if (fast) accumulate<NV, SIG>(p, pv, pc.ptr, id);
#if !AB_INGEST_PREFETCH
      if (i + THREADS < cnt) {
        if (keyed) nkey = __ldcs(ldg_ptr(&sg->key) + base + i + THREADS);
        nts = __ldcs(ldg_ptr(&sg->ts) + base + i + THREADS);
#pragma unroll
        for (int x = 0; x < NV; ++x) nv[x] = __ldcs(ldg_ptr(&sg->val[x]) + base + i + THREADS);
      }
#endif
    }
  }

  // per-pane on-time row counts: one atomic per (warp, pane) after a warp-level combine
  __syncwarp();
  flush_counts(p, pc, lane);
  // bookkeeping counters: warp reduce -> shared -> the last warp of the block publishes
  unsigned long long wl = late;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    wl += __shfl_xor_sync(0xffffffffu, wl, o);
    maxq = max(maxq, __shfl_xor_sync(0xffffffffu, maxq, o));
  }
  if (lane == 0) {
    if (wl) atomicAdd(&s_late, wl);
    if (maxq) atomicMax(&s_maxq, (unsigned long long)maxq);
    __threadfence_block();
    if (atomicAdd(&s_done, 1u) == THREADS / 32 - 1) {
      __threadfence_block();
      const unsigned long long bl = *(volatile unsigned long long*)&s_late;
      const unsigned long long mq = *(volatile unsigned long long*)&s_maxq;
      if (bl) atomicAdd(&p.counters->late_rows, bl);
      if (mq) atomicMax(&p.counters->max_q, mq);
    }
  }
}

#include "ingest_two_pass.cuh"

// Restore: merge a partial-state batch (AggregateExec(Partial) output written at a checkpoint,
// sliding_aggregating_window.rs:725-733) into one pane block.
struct PartialParams {
  const long long* key;
  const unsigned long long* state[MAX_ACC];  // state[0] = rows
  long long n;
  int keyed;
  int n_acc;
  int acc_kind[MAX_ACC];
  BDict dict;
  unsigned long long* pane;
  unsigned long long id_cap;
  Counters* counters;
};

__global__ void ingest_partial_kernel(const __grid_constant__ PartialParams p) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < p.n; i += stride) {
    uint32_t id = 0;
    if (p.keyed) {
      id = bd_lookup_or_insert(p.dict, p.key[i]);
      if (id >= ID_OVERFLOW) {
        atomicAdd(&p.counters->lost, 1ull);
        continue;
      }
    }
    for (int a = 0; a < p.n_acc; ++a) {
      unsigned long long* dst = p.pane + (unsigned long long)a * p.id_cap + id;
      unsigned long long v = p.state[a][i];
      switch (p.acc_kind[a]) {
        case ACC_ROWS:
        case ACC_SUM_I64:
          atomicAdd(dst, v);
          break;
        case ACC_SUM_F64:
          atomicAdd(reinterpret_cast<double*>(dst), __longlong_as_double((long long)v));
          break;
        case ACC_MIN_I64:
          atomicMin(reinterpret_cast<long long*>(dst), (long long)v);
          break;
        case ACC_MAX_I64:
          atomicMax(reinterpret_cast<long long*>(dst), (long long)v);
          break;
      }
    }
  }
}

// -------------------------------------------------------------------------------------------
// emission: pane merge (K4) + finalise + projection (K5) + compaction
// -------------------------------------------------------------------------------------------
constexpr int EMIT_INLINE = 16;
struct EmitParams {
  const unsigned long long* const* panes;  // device array of n_panes block pointers (more than EMIT_INLINE panes)
  const unsigned long long* inline_panes[EMIT_INLINE];  // ... or the pointers themselves
  int panes_inline;
  int n_panes;
  int n_acc;
  unsigned long long id_cap;
  uint32_t n_ids;
  int keyed;
  int acc_kind[MAX_ACC];
  // Output columns are attached to the accumulator they are computed from (no dynamic indexing in the
  // kernel): out_raw[a] receives the accumulator as is (COUNT(*) from a = 0, SUM / MIN / MAX), out_avg[a]
  // receives accumulator / rows as f64 (AVG).
  unsigned long long* out_raw[MAX_ACC];
  unsigned long long* out_avg[MAX_ACC];
  const long long* id_keys;
  long long* out_key;
  long long* out_wstart;
  long long* out_wend;
  long long* out_ts;
  long long wstart, wend, ts;
  unsigned int* out_count;  // cumulative over the operator's life (wraps); this emission's rows start at out_base
  unsigned int out_base;
  // running-window mode: W (same layout as a pane) is updated in place with
  // W += add panes, W -= sub panes and the output is produced from W.
  unsigned long long* running;
  int n_add;  // panes[0 .. n_add) enter, panes[n_add .. n_panes) leave
  // partial-state mode (checkpoint): emit raw accumulator columns instead of finalised aggregates
  int partial;
  unsigned long long* out_state[MAX_ACC];
};

constexpr int EMIT_THREADS = 256;

__device__ __forceinline__ unsigned long long merge_acc(int kind, unsigned long long a, unsigned long long v) {
  switch (kind) {
    case ACC_SUM_F64:
      return (unsigned long long)__double_as_longlong(__longlong_as_double((long long)a) + __longlong_as_double((long long)v));
    case ACC_MIN_I64: return (unsigned long long)min((long long)a, (long long)v);
    case ACC_MAX_I64: return (unsigned long long)max((long long)a, (long long)v);
    default: return a + v;  // ACC_ROWS, ACC_SUM_I64 (wrapping)
  }
}
__device__ __forceinline__ unsigned long long unmerge_acc(int kind, unsigned long long a, unsigned long long v) {
  if (kind == ACC_SUM_F64)
    return (unsigned long long)__double_as_longlong(__longlong_as_double((long long)a) - __longlong_as_double((long long)v));
  return a - v;
}

// Finalises and writes one output row (K4 finalise + K5 projection).
template <int NACC>
__device__ __forceinline__ void emit_row(const EmitParams& p, unsigned int o, const unsigned long long (&acc)[NACC],
                                         long long key) {
  const unsigned long long rows = acc[0];
  if (p.keyed) p.out_key[o] = key;
  if (p.partial) {
#pragma unroll
    for (int a = 0; a < NACC; ++a)
      p.out_state[a][o] = acc[a];
    p.out_ts[o] = p.ts;
    return;
  }
#pragma unroll
  for (int a = 0; a < NACC; ++a) {
    if (p.out_raw[a]) p.out_raw[a][o] = acc[a];
    if (p.out_avg[a]) {
      // f64 accumulator: sum of inputs cast to f64 (DataFusion's AVG state); integer accumulator: the exact
      // sum, converted once (guarded against overflow on ingest)
      const double num = p.acc_kind[a] == ACC_SUM_F64 ? __longlong_as_double((long long)acc[a]) : (double)(long long)acc[a];
      p.out_avg[a][o] = (unsigned long long)__double_as_longlong(num / (double)rows);
    }
  }
  if (p.out_wstart) {
    p.out_wstart[o] = p.wstart;
    p.out_wend[o] = p.wend;
  }
  p.out_ts[o] = p.ts;
}

// Two consecutive dense ids per thread: every accumulator array is read and written with 128-bit
// accesses; the block compacts its valid rows with two ballots per warp and one atomic per block.
template <bool RUNNING, int NACC>
__global__ void __launch_bounds__(EMIT_THREADS) emit_kernel(const __grid_constant__ EmitParams p) {
  __shared__ unsigned int s_warp[EMIT_THREADS / 32];
  __shared__ unsigned int s_base;
  const int tid = threadIdx.x;
  const int lane = tid & 31, w = tid >> 5;
  const uint32_t n_pairs = (p.n_ids + 1) / 2;
  const uint32_t n_iter = (n_pairs + EMIT_THREADS - 1) / EMIT_THREADS;
  for (uint32_t it = blockIdx.x; it < n_iter; it += gridDim.x) {
    const uint32_t pair = it * EMIT_THREADS + tid;
    const uint32_t id = pair * 2;
    unsigned long long acc0[NACC], acc1[NACC];
#pragma unroll
    for (int a = 0; a < NACC; ++a) {
      acc0[a] = 0;
      acc1[a] = 0;
    }
    const bool in0 = id < p.n_ids, in1 = id + 1 < p.n_ids;
    if (in0) {
      if (RUNNING) {
#pragma unroll
        for (int a = 0; a < NACC; ++a)
          {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(p.running + (unsigned long long)a * p.id_cap + id);
            acc0[a] = v.x;
            acc1[a] = v.y;
          }
        for (int k = 0; k < p.n_panes; ++k) {
          const unsigned long long* pane = p.panes_inline ? p.inline_panes[k] : p.panes[k];
          const bool add = k < p.n_add;
#pragma unroll
          for (int a = 0; a < NACC; ++a)
            {
              const ulonglong2 v = __ldcs(reinterpret_cast<const ulonglong2*>(pane + (unsigned long long)a * p.id_cap + id));
              const int kind = p.acc_kind[a];
              acc0[a] = add ? merge_acc(kind, acc0[a], v.x) : unmerge_acc(kind, acc0[a], v.x);
              acc1[a] = add ? merge_acc(kind, acc1[a], v.y) : unmerge_acc(kind, acc1[a], v.y);
            }
        }
        // a key that left the window restarts from exactly zero (no f64 drift carried over)
        const bool z0 = acc0[0] == 0, z1 = acc1[0] == 0;
#pragma unroll
        for (int a = 0; a < NACC; ++a)
          {
            if (z0) acc0[a] = 0;
            if (z1) acc1[a] = 0;
            *reinterpret_cast<ulonglong2*>(p.running + (unsigned long long)a * p.id_cap + id) = make_ulonglong2(acc0[a], acc1[a]);
          }
      } else {
#pragma unroll
        for (int a = 0; a < NACC; ++a)
          {
            unsigned long long ident = 0;
            if (p.acc_kind[a] == ACC_MIN_I64) ident = (unsigned long long)LLONG_MAX;
            if (p.acc_kind[a] == ACC_MAX_I64) ident = (unsigned long long)LLONG_MIN;
            acc0[a] = ident;
            acc1[a] = ident;
          }
        for (int k = 0; k < p.n_panes; ++k) {
          const unsigned long long* pane = p.panes_inline ? p.inline_panes[k] : p.panes[k];
#pragma unroll
          for (int a = 0; a < NACC; ++a)
            {
              const ulonglong2 v = __ldcs(reinterpret_cast<const ulonglong2*>(pane + (unsigned long long)a * p.id_cap + id));
              const int kind = p.acc_kind[a];
              acc0[a] = merge_acc(kind, acc0[a], v.x);
              acc1[a] = merge_acc(kind, acc1[a], v.y);
            }
        }
      }
    }
    const bool v0 = in0 && acc0[0] != 0, v1 = in1 && acc1[0] != 0;
    const unsigned int b0 = __ballot_sync(0xffffffffu, v0), b1 = __ballot_sync(0xffffffffu, v1);
    if (lane == 0) s_warp[w] = __popc(b0) + __popc(b1);
    __syncthreads();
    if (tid == 0) {
      unsigned int total = 0;
      for (int i = 0; i < EMIT_THREADS / 32; ++i) {
        unsigned int c = s_warp[i];
        s_warp[i] = total;
        total += c;
      }
      s_base = total ? atomicAdd(p.out_count, total) - p.out_base : 0u;
    }
    __syncthreads();
    const unsigned int lt = (1u << lane) - 1u;
    const unsigned int o0 = s_base + s_warp[w] + __popc(b0 & lt) + __popc(b1 & lt);
    ulonglong2 keys = make_ulonglong2(0, 0);
    if ((v0 || v1) && p.keyed) keys = *reinterpret_cast<const ulonglong2*>(p.id_keys + id);
    if (v0) emit_row<NACC>(p, o0, acc0, (long long)keys.x);
    if (v1) emit_row<NACC>(p, o0 + (v0 ? 1u : 0u), acc1, (long long)keys.y);
    __syncthreads();
  }
}

// checkpoint fold: frozen += active; active = identity  (see Pane::frozen)
struct FoldParams {
  unsigned long long* active;
  unsigned long long* frozen;
  unsigned long long id_cap;
  uint32_t n_ids;
  int n_acc;
  int acc_kind[MAX_ACC];
};
__global__ void fold_kernel(const __grid_constant__ FoldParams p) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t stride = gridDim.x * blockDim.x;
  for (; i < p.n_ids; i += stride) {
    for (int a = 0; a < p.n_acc; ++a) {
      unsigned long long* fa = p.frozen + (unsigned long long)a * p.id_cap + i;
      unsigned long long* aa = p.active + (unsigned long long)a * p.id_cap + i;
      unsigned long long f = *fa, v = *aa, ident = 0;
      switch (p.acc_kind[a]) {
        case ACC_ROWS:
        case ACC_SUM_I64:
          f += v;
          break;
        case ACC_SUM_F64:
          f = (unsigned long long)__double_as_longlong(__longlong_as_double((long long)f) +
                                                       __longlong_as_double((long long)v));
          break;
        case ACC_MIN_I64:
          f = (unsigned long long)min((long long)f, (long long)v);
          ident = (unsigned long long)LLONG_MAX;
          break;
        case ACC_MAX_I64:
          f = (unsigned long long)max((long long)f, (long long)v);
          ident = (unsigned long long)LLONG_MIN;
          break;
      }
      *fa = f;
      *aa = ident;
    }
  }
}

// -------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------
struct Pane {
  int64_t bin = 0;
  unsigned long long* dev = nullptr;     // active accumulators (receives REDs)
  unsigned long long* frozen = nullptr;  // state already written to a checkpoint / restored
  int slot = -1;
  bool in_tier = false;
  uint64_t rows = 0;  // on-time rows aggregated into this pane
  bool exported = false;  // its state is already in the shim's state table (checkpointed / restored)
  bool delta_exported = false;  // `frozen` is in the state table; only `dev` is new
};

struct LaunchRec {
  cudaEvent_t done = nullptr;
  cudaEvent_t t0 = nullptr, t1 = nullptr;
  Counters* h_counters = nullptr;  // pinned: [Counters | slot_rows[MAX_RING]] as copied back in one piece
  unsigned long long* h_slot_rows = nullptr;
  uint64_t rows = 0;
  bool in_flight = false;
  int chunk = -1;  // staging chunk read by this launch (-1: none)
};

constexpr size_t RELEASE_GROUP = 16;
struct PendingRelease {
  cudaEvent_t ev;
  std::vector<ArrowArray> arrs;  // moved-in copies; released when ev completes
};

class WindowAggOp final : public OpBase {
 public:
  explicit WindowAggOp(const ArroyoB200OpConfig& c);
  ~WindowAggOp() override;

  void on_start(ArrowArray* state, ArrowSchema* schemas, int64_t n, int64_t watermark, int64_t table_min) override;
  void process_batch(uint32_t, uint32_t, ArrowArray* batch, const ArrowSchema* schema) override;
  void process_device_batch(uint32_t, uint32_t, const uint64_t* cols, int32_t n_cols, int64_t n_rows) override;
  void handle_watermark(int64_t wm, BatchesPriv* out_host, std::vector<ArroyoB200DeviceBatch>* out_dev) override;
  void handle_checkpoint(int64_t wm, BatchesPriv* out) override;
  void on_close(int, BatchesPriv*) override { flush(); }
  void flush() override;
  void submit() override;
  void begin_watermark(int64_t wm) override;
  bool poll_watermark(bool block) override;
  void begin_watermark_device(int64_t wm) override;
  void poll_watermark_device(std::vector<ArroyoB200DeviceBatch>* out) override;
  void stats(ArroyoB200Stats* out) override;

 private:
  // config-derived
  bool sliding_;
  int64_t width_, slide_;  // slide_ == width_ for tumbling
  bool keyed_;
  int key_col_, ts_col_;
  int n_vals_ = 0;
  int val_cols_[MAX_VALS];
  int n_acc_ = 1;
  int acc_kind_[MAX_ACC];
  int acc_val_[MAX_ACC];
  int n_aggs_;
  int agg_kind_[ARROYO_B200_MAX_AGGS];
  int agg_acc_[ARROYO_B200_MAX_AGGS];
  bool invertible_ = true;
  // AVG(Int64) from the exact integer sum instead of a separate f64 RED per row (one scattered access
  // less per row).  Valid while no per-key sum can overflow i64: every guarded value is < 2^31 in
  // magnitude (checked per row on the device) and no window holds 2^32 rows (checked on the host);
  // otherwise the operator promotes itself to f64 accumulators (promote_avg).  The result differs from
  // DataFusion's running f64 sum by at most n * 2^-53 relative (north-star tolerance: 1e-6).
  bool avg_exact_ = true;
  unsigned int guard_vals_ = 0;
  int rows_slot_ = -1;  // value slot of the carried row count (partial-aggregate inputs)
  bool running_mode_ = false;
  bool profile_;
  std::string key_format_ = "l";
  std::vector<std::string> agg_format_;

  int device_;
  cudaStream_t stream_ = nullptr;
  bool own_stream_ = false;
  int num_sms_ = 148;

  // dictionary (bdict.cuh): n_buckets_ buckets of BD_KS slots; ids = BD_ID_BASE + bucket * BD_CAPB + index
  uint64_t id_cap_ = 0;
  uint64_t n_buckets_ = 1;
  DevBuf slots_, bucket_nkeys_, id_keys_;
  // bookkeeping the kernels report back, one contiguous buffer = one device->host copy per launch:
  // [Counters | slot_rows[MAX_RING]].  slot_rows (on-time rows per ring slot) is cumulative; the host works with the
  // difference between consecutive launches (no per-launch memset).
  DevBuf book_;
  static constexpr size_t BOOK_SLOT_OFF = (sizeof(Counters) + 15) / 16 * 16;
  Counters* d_counters() const { return reinterpret_cast<Counters*>(book_.p); }
  unsigned long long* d_slot_rows() const { return reinterpret_cast<unsigned long long*>((char*)book_.p + BOOK_SLOT_OFF); }
  std::vector<unsigned long long> slot_rows_seen_;
  uint32_t n_keys_host_ = 1;       // ids in use = the id range the element-wise kernels walk (all of it: bucket ranges)
  uint32_t total_keys_host_ = 0;   // keys in the dictionary (statistics, growth policy)
  uint32_t dict_full_seen_ = 0;
  // two-pass ingest (ingest_two_pass.cuh)
  DevBuf part_, part_cursor_;  // part_cursor_: two cursor sets; a launch's aggregation pass re-zeroes the other one
  uint32_t part_cap_ = 0;
  int part_flip_ = 0;
  bool two_pass_attr_set_ = false;
  bool two_pass_enabled_ = true;
  uint64_t part_overflow_seen_ = 0;
  mutable int two_pass_pause_ = 0;  // launches left on the one-pass kernel after a skewed launch
  bool two_pass_eligible(uint64_t rows) const;
  void launch_two_pass(IngestParams& p, uint64_t rows, long long tiles_direct);
  BDict dict_view() const;
  // asynchronous emission (begin_watermark / poll_watermark): windows are copied back on a second stream so the
  // device->host traffic overlaps the host->device traffic of the batches that follow
  cudaStream_t out_stream_ = nullptr;
  cudaEvent_t emit_done_ = nullptr, out_done_ = nullptr;
  bool async_out_ = false, out_inflight_ = false;
  void wait_outputs();
  static constexpr size_t COPY_GROUP = 48;
  std::vector<void*> copy_dst_, copy_src_;
  std::vector<size_t> copy_size_;
  bool batch_copy_ok_ = true;
  void queue_copy(void* dst, const void* src, size_t bytes);
  void flush_copies();
  std::vector<ArrowArray> open_release_;  // staged inputs whose copies have no release event yet
  std::vector<cudaEvent_t> ev_pool_;
  void seal_release();

  // ring
  uint32_t ring_ = 16;
  std::vector<long long> h_pane_bins_;
  std::vector<unsigned long long*> h_pane_ptrs_;
  DevBuf d_pane_bins_, d_pane_ptrs_;
  bool ring_dirty_ = true;
  std::map<int64_t, Pane> panes_;
  std::vector<std::pair<unsigned long long*, uint64_t>> free_panes_;  // (block, dirty ids)
  std::vector<DevBuf> pane_storage_;
  int64_t late_bin_ = LLONG_MIN;
  int64_t max_bin_seen_ = LLONG_MIN;

  // running window block
  unsigned long long* running_ = nullptr;
  std::set<int64_t> in_running_;
  std::map<int64_t, Pane> zombies_;  // left the store; blocks kept until the next emit subtracts them

  // planners
  std::unique_ptr<TumblingPlanner> tumbling_;
  std::unique_ptr<SlidingPlanner> sliding_planner_;

  // staging
  static constexpr int NCHUNK = 3;
  static constexpr int NLAUNCH = 3;
  int64_t chunk_rows_ = 1 << 24;  // rows per ingest launch: one headline pane; fixed per-launch costs (table builds, tails) halve vs 2^23
  // device-resident batches are only pointers: they may pile up a little past one chunk before a launch is forced, so a
  // stream whose watermarks arrive every chunk_rows_ rows or so gets one launch per watermark instead of a chunk-sized
  // launch plus a fragment
  int64_t launch_rows_ = (1 << 24) + (1 << 22);
  DevBuf chunk_[NCHUNK];
  cudaEvent_t chunk_free_[NCHUNK] = {nullptr, nullptr, nullptr};
  // host batches are staged by the copy engine on their own stream, so the link never waits for an ingest kernel:
  // copy stream --copied_--> compute stream (kernel reads the chunk) --chunk_free_--> copy stream (chunk reused)
  cudaStream_t copy_stream_ = nullptr;
  cudaEvent_t copied_ = nullptr;
  int cur_chunk_ = 0;
  int64_t cur_rows_ = 0;
  std::vector<Segment> segs_;
  int64_t pending_rows_ = 0;
  bool pending_uses_chunk_ = false;
  PinnedBuf h_segs_[NLAUNCH];
  DevBuf d_segs_[NLAUNCH];
  LaunchRec launches_[NLAUNCH];
  PinnedBuf h_book_[NLAUNCH];
  int next_launch_ = 0;
  std::deque<int> in_flight_;
  std::deque<PendingRelease> releases_;
  std::vector<ArrowArray> zero_copy_inputs_;  // pinned input batches read in place by the next launch

  // deferred rows (two sets: one being filled, one being re-ingested)
  uint64_t defer_cap_ = 0;
  DevBuf defer_[2][2 + MAX_VALS];
  int defer_cur_ = 0;
  Counters last_counters_{};
  bool have_counters_ = false;
  bool draining_ = false;
  bool need_promote_ = false;

  // emission output
  struct OutSet {
    DevBuf key, wstart, wend, ts;
    DevBuf agg[ARROYO_B200_MAX_AGGS];
    DevBuf state[MAX_ACC];
    uint64_t cap = 0;
  };
  std::vector<std::unique_ptr<OutSet>> out_sets_;
  DevBuf d_emit_panes_, d_out_count_;
  unsigned int out_count_base_ = 0;
  PinnedBuf h_out_count_;
  // deferred row counts (begin_watermark_device / poll_watermark_device): the emission is enqueued without waiting
  // for its windows' row counts, which travel to these pinned slots; `pending_dev[i].n_rows` = -(slot + 1) until
  // resolve_deferred() has read them
  static constexpr int COUNT_SLOTS = 64;
  PinnedBuf h_out_counts_;
  bool defer_counts_ = false;
  int count_slots_used_ = 0;
  bool counts_pending_ = false;
  cudaEvent_t counts_done_ = nullptr;
  void resolve_deferred();

  ArroyoB200Stats st_{};
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> emit_events_;  // pooled: [0, emit_events_used_) are recorded
  size_t emit_events_used_ = 0;

  // helpers
  void set_device() { AB_CUDA(cudaSetDevice(device_)); }
  void alloc_dictionary(uint64_t n_buckets);
  void preallocate();
  void grow_ids();
  void apply_l2_policy();
  void promote_avg();
  void relayout_blocks(int old_n_acc, const std::vector<std::pair<int, int>>& f64_from);
  unsigned long long* acquire_block();
  void release_block(unsigned long long* blk);
  void init_block(unsigned long long* blk, uint64_t n_ids);
  void ensure_pane(int64_t bin);
  void drop_pane(int64_t bin);
  void upload_ring();
  void add_segment(const long long* key, const long long* ts, const long long* const* vals, int64_t n);
  void launch_pending();
  void launch_segments(const std::vector<Segment>& segs, int chunk);
  void absorb(int li);
  void sync_all();
  void drain_deferred();
  void poll_releases(bool wait);
  void rotate_chunk();
  void touch(int64_t bin);
  OutSet* out_set(size_t i, uint64_t cap);
  int64_t run_emit(const std::vector<const unsigned long long*>& blocks, int n_add, bool use_running, bool partial,
                   int64_t wstart, int64_t wend, int64_t ts, OutSet* os);
  void emit_window(int64_t a, int64_t b, size_t out_index, BatchesPriv* out_host,
                   std::vector<ArroyoB200DeviceBatch>* out_dev);
  void export_window(OutSet* os, int64_t n, BatchesPriv* out_host);
  void export_partial(OutSet* os, int64_t n, BatchesPriv* out);
  void collect_emit_times();
  void lookahead();
};

WindowAggOp::WindowAggOp(const ArroyoB200OpConfig& c) {
  cfg = c;
  sliding_ = c.kind == ARROYO_B200_SLIDING_AGGREGATE;
  name = sliding_ ? "sliding_window" : "tumbling_window";
  AB_REQUIRE(c.width_ns > 0, ARROYO_B200_UNSUPPORTED, "width_micros == 0 (instant window) is not supported");
  width_ = c.width_ns;
  slide_ = sliding_ ? c.slide_ns : c.width_ns;
  AB_REQUIRE(slide_ >= 2, ARROYO_B200_INVALID_ARGUMENT, "slide must be >= 2 ns");
  if (sliding_)
    AB_REQUIRE(width_ % slide_ == 0, ARROYO_B200_INVALID_ARGUMENT,
               "hop width must be a multiple of the slide (arroyo-planner/src/lib.rs:640-655)");
  AB_REQUIRE(c.n_key_cols == 0 || c.n_key_cols == 1, ARROYO_B200_UNSUPPORTED,
             "only 0 or 1 group-by key columns are supported");
  keyed_ = c.n_key_cols == 1;
  key_col_ = c.key_col;
  ts_col_ = c.timestamp_col;
  AB_REQUIRE(c.n_cols >= 1 && c.n_cols <= ARROYO_B200_MAX_COLS, ARROYO_B200_INVALID_ARGUMENT, "bad n_cols");
  AB_REQUIRE(ts_col_ >= 0 && ts_col_ < c.n_cols, ARROYO_B200_INVALID_ARGUMENT, "bad timestamp_col");
  AB_REQUIRE(!keyed_ || (key_col_ >= 0 && key_col_ < c.n_cols), ARROYO_B200_INVALID_ARGUMENT, "bad key_col");
  AB_REQUIRE(c.n_aggs >= 1 && c.n_aggs <= ARROYO_B200_MAX_AGGS, ARROYO_B200_INVALID_ARGUMENT, "bad n_aggs");
  n_aggs_ = c.n_aggs;
  avg_exact_ = !(c.flags & ARROYO_B200_FLAG_AVG_F64);
  acc_kind_[0] = ACC_ROWS;
  acc_val_[0] = 0;
  for (int g = 0; g < n_aggs_; ++g) {
    int kind = c.aggs[g].kind;
    agg_kind_[g] = kind;
    agg_acc_[g] = 0;
    if (kind == ARROYO_B200_AGG_COUNT_STAR) {
      agg_format_.push_back("l");
      continue;
    }
    int col = c.aggs[g].input_col;
    AB_REQUIRE(col >= 0 && col < c.n_cols, ARROYO_B200_INVALID_ARGUMENT, "aggregate input column out of range");
    int vs = -1;
    for (int v = 0; v < n_vals_; ++v)
      if (val_cols_[v] == col) vs = v;
    if (vs < 0) {
      AB_REQUIRE(n_vals_ < MAX_VALS, ARROYO_B200_UNSUPPORTED, "more than 4 distinct aggregate input columns");
      vs = n_vals_;
      val_cols_[n_vals_++] = col;
    }
    int ak;
    switch (kind) {
      case ARROYO_B200_AGG_SUM_I64: ak = ACC_SUM_I64; agg_format_.push_back("l"); break;
      case ARROYO_B200_AGG_AVG_I64:
        // exact mode: AVG shares the wrapping integer sum and is finalised as (double)sum / count
        ak = avg_exact_ ? ACC_SUM_I64 : ACC_SUM_F64;
        if (avg_exact_) guard_vals_ |= 1u << vs;
        agg_format_.push_back("g");
        break;
      case ARROYO_B200_AGG_MIN_I64: ak = ACC_MIN_I64; agg_format_.push_back("l"); invertible_ = false; break;
      case ARROYO_B200_AGG_MAX_I64: ak = ACC_MAX_I64; agg_format_.push_back("l"); invertible_ = false; break;
      default:
        throw Error(ARROYO_B200_UNSUPPORTED, "unsupported aggregate kind");
    }
    // share accumulators between identical (kind, column) pairs
    int found = -1;
    for (int a = 1; a < n_acc_; ++a)
      if (acc_kind_[a] == ak && acc_val_[a] == vs) found = a;
    if (found < 0) {
      found = n_acc_;
      acc_kind_[n_acc_] = ak;
      acc_val_[n_acc_] = vs;
      ++n_acc_;
    }
    agg_acc_[g] = found;
  }
  if (c.partial_count_col_plus1 > 0) {
    const int col = c.partial_count_col_plus1 - 1;
    AB_REQUIRE(col < c.n_cols, ARROYO_B200_INVALID_ARGUMENT, "partial count column out of range");
    int vs = -1;
    for (int v = 0; v < n_vals_; ++v)
      if (val_cols_[v] == col) vs = v;
    if (vs < 0) {
      AB_REQUIRE(n_vals_ < MAX_VALS, ARROYO_B200_UNSUPPORTED, "more than 4 distinct aggregate input columns");
      vs = n_vals_;
      val_cols_[n_vals_++] = col;
    }
    rows_slot_ = vs;
    // partial sums are not bounded by 2^31: exactness of the integer AVG path rests on the upstream
    // (raw-row) stage's guard and on the window row bound checked at emission
    guard_vals_ = 0;
  }
  profile_ = (c.flags & ARROYO_B200_FLAG_PROFILE) != 0;
  // The running window W += entering - leaving is used only while every accumulator is exactly invertible
  // (row counts, wrapping integer sums).  An f64 accumulator would carry cancellation error from rows that
  // have left the window (measured: 1e-5 relative after a 2^61 value passed through), so those
  // configurations re-merge the panes of each window like the reference does.
  bool has_f64 = false;
  for (int a = 1; a < n_acc_; ++a) has_f64 = has_f64 || acc_kind_[a] == ACC_SUM_F64;
  running_mode_ = sliding_ && invertible_ && !has_f64 && !(c.flags & ARROYO_B200_FLAG_REMERGE_ONLY) && width_ > slide_;

  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0)
    throw Error(ARROYO_B200_FATAL, "no CUDA device available: libarroyo_b200 has no CPU fallback");
  device_ = c.device;
  AB_REQUIRE(device_ >= 0 && device_ < count, ARROYO_B200_INVALID_ARGUMENT, "bad device ordinal");
  set_device();
  cudaDeviceProp prop{};
  AB_CUDA(cudaGetDeviceProperties(&prop, device_));
  num_sms_ = prop.multiProcessorCount;
  if (c.stream) {
    stream_ = (cudaStream_t)c.stream;
  } else {
    AB_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    own_stream_ = true;
  }

  if (sliding_) sliding_planner_.reset(new SlidingPlanner(width_, slide_));
  else tumbling_.reset(new TumblingPlanner(width_));

  book_.alloc(BOOK_SLOT_OFF + MAX_RING * sizeof(unsigned long long));
  AB_CUDA(cudaMemsetAsync(book_.p, 0, book_.bytes, stream_));
  slot_rows_seen_.assign(MAX_RING, 0);
  Counters init{};
  init.max_q = 0;
  init.n_keys = 0;
  AB_CUDA(cudaMemcpyAsync(book_.p, &init, sizeof init, cudaMemcpyHostToDevice, stream_));
  last_counters_ = init;

  // one bucket per ~BD_MEAN expected keys (the bucket count doubles when a bucket runs out of ids)
  uint64_t want = c.expected_keys ? c.expected_keys : (1ull << 16);
  alloc_dictionary(keyed_ ? bd_buckets_for(want) : 1);
  {
    const char* e = getenv("ARROYO_B200_NO_TWO_PASS");
    two_pass_enabled_ = !(e && atoi(e) != 0) && !(c.flags & ARROYO_B200_FLAG_NO_TWO_PASS);
  }

  h_pane_bins_.assign(MAX_RING, FREE_BIN);
  h_pane_ptrs_.assign(MAX_RING, nullptr);
  d_pane_bins_.alloc(MAX_RING * sizeof(long long));
  d_pane_ptrs_.alloc(MAX_RING * sizeof(void*));
  if (sliding_) {
    uint64_t need = (uint64_t)(width_ / slide_) + 8;
    while (ring_ < need && ring_ < MAX_RING) ring_ <<= 1;
  }

  const int n_used = 2 + n_vals_;
  for (int i = 0; i < NCHUNK; ++i) {
    AB_CUDA(cudaEventCreateWithFlags(&chunk_free_[i], cudaEventDisableTiming));
    if (i == 0) {
      AB_CUDA(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
      AB_CUDA(cudaEventCreateWithFlags(&copied_, cudaEventDisableTiming));
    }
  }
  (void)n_used;
  for (int i = 0; i < NLAUNCH; ++i) {
    h_segs_[i].alloc(MAX_SEGS * sizeof(Segment));
    d_segs_[i].alloc(MAX_SEGS * sizeof(Segment));
    h_book_[i].alloc(BOOK_SLOT_OFF + MAX_RING * sizeof(unsigned long long));
    launches_[i].h_counters = h_book_[i].as<Counters>();
    launches_[i].h_slot_rows = reinterpret_cast<unsigned long long*>((char*)h_book_[i].p + BOOK_SLOT_OFF);
    AB_CUDA(cudaEventCreateWithFlags(&launches_[i].done, cudaEventDisableTiming));
    if (profile_) {
      AB_CUDA(cudaEventCreate(&launches_[i].t0));
      AB_CUDA(cudaEventCreate(&launches_[i].t1));
    }
  }
  if (c.reserved >= 16 && c.reserved <= 26) chunk_rows_ = 1ll << c.reserved;  // rows per ingest launch (default 2^24)
  launch_rows_ = chunk_rows_ + chunk_rows_ / 4;
  defer_cap_ = (uint64_t)launch_rows_ * 2;
  d_emit_panes_.alloc(MAX_MERGE * sizeof(void*));
  d_out_count_.alloc(sizeof(unsigned int));
  AB_CUDA(cudaMemsetAsync(d_out_count_.p, 0, sizeof(unsigned int), stream_));
  h_out_count_.alloc(sizeof(unsigned int));
  h_out_counts_.alloc(COUNT_SLOTS * sizeof(unsigned int));
  preallocate();
  AB_CUDA(cudaStreamSynchronize(stream_));
}

// Everything the steady state needs is allocated when the operator is created: the panes of one full window
// plus the look-ahead panes, the running-window block, one set of deferred-row columns and two output sets.
// cudaMalloc inside process_batch / handle_watermark serialises the device and showed up as milliseconds per
// step in short runs (the driver's 5-warm-up / 20-step scaling runs timed little else).
void WindowAggOp::preallocate() {
  const size_t block_bytes = (size_t)n_acc_ * id_cap_ * sizeof(unsigned long long);
  size_t want = (sliding_ ? (size_t)(width_ / slide_) : 1) + 4 + (running_mode_ ? 1 : 0);
  const size_t budget = (size_t)4 << 30;
  want = std::min<size_t>(std::min<size_t>(want, 64), std::max<size_t>(budget / std::max<size_t>(block_bytes, 1), 4));
  for (size_t i = 0; i < want; ++i) {
    pane_storage_.emplace_back(block_bytes);
    auto* blk = pane_storage_.back().as<unsigned long long>();
    init_block(blk, id_cap_);
    free_panes_.emplace_back(blk, 0);  // already holds the identity: nothing to reset when it is acquired
  }
  for (int c = 0; c < 2 + n_vals_; ++c) defer_[0][c].alloc(defer_cap_ * 8);
  out_set(0, id_cap_);
  out_set(1, id_cap_);
}

WindowAggOp::~WindowAggOp() {
  cudaSetDevice(device_);
  if (counts_done_) cudaEventDestroy(counts_done_);
  // nothing may still be reading the input batches or writing output buffers when they are handed back
  if (copy_stream_) cudaStreamSynchronize(copy_stream_);
  if (out_stream_) cudaStreamSynchronize(out_stream_);
  cudaStreamSynchronize(stream_);
  for (auto& r : releases_) {
    for (auto& a : r.arrs)
      if (a.release) a.release(&a);
    cudaEventDestroy(r.ev);
  }
  for (auto& a : zero_copy_inputs_)
    if (a.release) a.release(&a);
  for (auto& a : open_release_)
    if (a.release) a.release(&a);
  for (auto e : ev_pool_) cudaEventDestroy(e);
  for (int i = 0; i < NCHUNK; ++i)
    if (chunk_free_[i]) cudaEventDestroy(chunk_free_[i]);
  if (copy_stream_) {
    cudaStreamSynchronize(copy_stream_);
    cudaStreamDestroy(copy_stream_);
    cudaEventDestroy(copied_);
  }
  for (int i = 0; i < NLAUNCH; ++i) {
    if (launches_[i].done) cudaEventDestroy(launches_[i].done);
    if (launches_[i].t0) cudaEventDestroy(launches_[i].t0);
    if (launches_[i].t1) cudaEventDestroy(launches_[i].t1);
  }
  for (auto& e : emit_events_) {
    cudaEventDestroy(e.first);
    cudaEventDestroy(e.second);
  }
  if (out_stream_) {
    cudaStreamSynchronize(out_stream_);
    cudaStreamDestroy(out_stream_);
    cudaEventDestroy(emit_done_);
    cudaEventDestroy(out_done_);
  }
  if (own_stream_ && stream_) cudaStreamDestroy(stream_);
}

void WindowAggOp::alloc_dictionary(uint64_t n_buckets) {
  n_buckets_ = n_buckets;
  id_cap_ = bd_id_cap(n_buckets_);
  AB_REQUIRE(id_cap_ < (1ull << 31), ARROYO_B200_RUNTIME, "key dictionary too large");
  n_keys_host_ = (uint32_t)(BD_ID_BASE + n_buckets_ * BD_CAPB);
  id_keys_.alloc(id_cap_ * sizeof(long long));
  bd_fill_keys_kernel<<<num_sms_ * 4, 256, 0, stream_>>>(id_keys_.as<long long>(), id_cap_);
  AB_CUDA(cudaGetLastError());
  bucket_nkeys_.alloc(n_buckets_ * sizeof(unsigned int));
  AB_CUDA(cudaMemsetAsync(bucket_nkeys_.p, 0, n_buckets_ * sizeof(unsigned int), stream_));
  if (keyed_) {
    slots_.alloc(n_buckets_ * BD_KS * sizeof(BSlot));
    bd_init_kernel<<<num_sms_ * 4, 256, 0, stream_>>>(slots_.as<BSlot>(), n_buckets_ * BD_KS);
    AB_CUDA(cudaGetLastError());
    ++st_.kernel_launches;
    apply_l2_policy();
  }
}

BDict WindowAggOp::dict_view() const {
  BDict d{};
  d.slots = slots_.as<BSlot>();
  d.nkeys = bucket_nkeys_.as<unsigned int>();
  d.id_keys = id_keys_.as<long long>();
  d.n_total = (unsigned int*)((char*)book_.p + offsetof(Counters, n_keys));
  d.n_buckets = (uint32_t)n_buckets_;
  return d;
}

// ARROYO_B200_L2_PERSIST=1: ask L2 to keep the key dictionary resident (persisting access-policy window on the
// operator's stream); everything else the stream touches is treated as streaming.
void WindowAggOp::apply_l2_policy() {
  const char* e = getenv("ARROYO_B200_L2_PERSIST");
  if (!e || atoi(e) == 0 || !slots_.p) return;
  int max_persist = 0, max_window = 0;
  cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, device_);
  cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, device_);
  size_t bytes = std::min<size_t>(n_buckets_ * BD_KS * sizeof(BSlot), (size_t)std::max(max_window, 0));
  if (bytes == 0 || max_persist <= 0) return;
  cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, std::min<size_t>(bytes, (size_t)max_persist));
  cudaStreamAttrValue attr{};
  attr.accessPolicyWindow.base_ptr = slots_.p;
  attr.accessPolicyWindow.num_bytes = bytes;
  attr.accessPolicyWindow.hitRatio = std::min(1.0f, (float)max_persist / (float)bytes);
  attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  cudaStreamSetAttribute(stream_, cudaStreamAttributeAccessPolicyWindow, &attr);
  cudaGetLastError();
}

void WindowAggOp::init_block(unsigned long long* blk, uint64_t n_ids) {
  if (n_ids == 0) return;
  InitParams ip{};
  ip.pane = blk;
  ip.id_cap = id_cap_;
  ip.n = n_ids;
  ip.n_acc = n_acc_;
  for (int a = 0; a < n_acc_; ++a) ip.acc_kind[a] = acc_kind_[a];
  int blocks = (int)std::min<uint64_t>((n_ids + 255) / 256, (uint64_t)num_sms_ * 8);
  pane_init_kernel<<<blocks, 256, 0, stream_>>>(ip);
  AB_CUDA(cudaGetLastError());
  ++st_.kernel_launches;
}

unsigned long long* WindowAggOp::acquire_block() {
  if (!free_panes_.empty()) {
    auto pr = free_panes_.back();
    free_panes_.pop_back();
    init_block(pr.first, pr.second);
    return pr.first;
  }
  pane_storage_.emplace_back((size_t)n_acc_ * id_cap_ * sizeof(unsigned long long));
  auto* blk = pane_storage_.back().as<unsigned long long>();
  init_block(blk, id_cap_);
  return blk;
}

void WindowAggOp::release_block(unsigned long long* blk) {
  if (!blk) return;
  free_panes_.emplace_back(blk, std::min<uint64_t>(id_cap_, (uint64_t)n_keys_host_ + 1));
}

// new[a][map[i]] = old[a][i] for every old id that holds a key
__global__ void permute_block_kernel(const unsigned long long* __restrict__ old_blk, unsigned long long* __restrict__ new_blk,
                                     const uint32_t* __restrict__ map, uint32_t old_ids, uint64_t old_cap, uint64_t new_cap,
                                     int n_acc) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (; i < old_ids; i += stride) {
    const uint32_t m = map[i];
    if (m == ID_UNSET || m >= ID_OVERFLOW) continue;
    for (int a = 0; a < n_acc; ++a) new_blk[(uint64_t)a * new_cap + m] = old_blk[(uint64_t)a * old_cap + i];
  }
}

// Doubles the bucket count: every key is re-inserted into the new dictionary (its id changes), and every live pane
// block is permuted with the old -> new id map.
void WindowAggOp::grow_ids() {
  AB_REQUIRE(keyed_, ARROYO_B200_RUNTIME, "grow_ids on an unkeyed aggregate");
  const uint64_t old_cap = id_cap_;
  const uint32_t old_ids = n_keys_host_;
  BDict old_d = dict_view();
  DevBuf old_slots = std::move(slots_), old_nkeys = std::move(bucket_nkeys_), old_keys = std::move(id_keys_);
  old_d.slots = old_slots.as<BSlot>();
  old_d.nkeys = old_nkeys.as<unsigned int>();
  old_d.id_keys = old_keys.as<long long>();
  const unsigned int zero = 0;
  AB_CUDA(cudaMemcpyAsync((char*)book_.p + offsetof(Counters, n_keys), &zero, sizeof zero, cudaMemcpyHostToDevice, stream_));
  alloc_dictionary(n_buckets_ * 2);
  const uint64_t new_cap = id_cap_;
  DevBuf map((size_t)old_cap * sizeof(uint32_t));
  {
    const int grid = (int)std::min<uint64_t>((old_ids + 255) / 256, (uint64_t)num_sms_ * 8);
    bd_rehash_kernel<<<std::max(grid, 1), 256, 0, stream_>>>(old_d, dict_view(), old_ids, map.as<uint32_t>());
    AB_CUDA(cudaGetLastError());
    ++st_.kernel_launches;
  }
  std::vector<DevBuf> new_storage;
  auto migrate = [&](unsigned long long* old_blk) -> unsigned long long* {
    if (!old_blk) return nullptr;
    new_storage.emplace_back((size_t)n_acc_ * new_cap * sizeof(unsigned long long));
    auto* nb = new_storage.back().as<unsigned long long>();
    init_block(nb, new_cap);
    const int grid = (int)std::min<uint64_t>((old_ids + 255) / 256, (uint64_t)num_sms_ * 8);
    permute_block_kernel<<<std::max(grid, 1), 256, 0, stream_>>>(old_blk, nb, map.as<uint32_t>(), old_ids, old_cap, new_cap,
                                                               n_acc_);
    AB_CUDA(cudaGetLastError());
    ++st_.kernel_launches;
    return nb;
  };
  for (auto& kv : panes_) {
    kv.second.dev = migrate(kv.second.dev);
    kv.second.frozen = migrate(kv.second.frozen);
    if (kv.second.slot >= 0) h_pane_ptrs_[kv.second.slot] = kv.second.dev;
  }
  for (auto& kv : zombies_) {
    kv.second.dev = migrate(kv.second.dev);
    kv.second.frozen = migrate(kv.second.frozen);
  }
  running_ = migrate(running_);
  Counters c{};
  AB_CUDA(cudaMemcpyAsync(&c, book_.p, sizeof c, cudaMemcpyDeviceToHost, stream_));
  AB_CUDA(cudaStreamSynchronize(stream_));
  total_keys_host_ = c.n_keys;
  free_panes_.clear();
  pane_storage_ = std::move(new_storage);
  // (output sets stay: a caller may still hold the last emission's device pointers; out_set() grows them on demand)
  part_cap_ = 0;      // the partition buffer is sized by the bucket count
  ring_dirty_ = true;
}

// fsum[id] = (double)(int64)sum[id]
__global__ void i64_to_f64_kernel(const unsigned long long* __restrict__ src, unsigned long long* __restrict__ dst, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) dst[i] = (unsigned long long)__double_as_longlong((double)(long long)src[i]);
}

// Re-creates every live block with the current n_acc_; accumulators [0, old_n_acc) are copied, and each
// (new index, source index) pair in f64_from is filled with the f64 image of the source integer sum.
void WindowAggOp::relayout_blocks(int old_n_acc, const std::vector<std::pair<int, int>>& f64_from) {
  std::vector<DevBuf> new_storage;
  const uint32_t n_valid = (uint32_t)std::min<uint64_t>(n_keys_host_, id_cap_);
  auto migrate = [&](unsigned long long* old_blk) -> unsigned long long* {
    if (!old_blk) return nullptr;
    new_storage.emplace_back((size_t)n_acc_ * id_cap_ * sizeof(unsigned long long));
    auto* nb = new_storage.back().as<unsigned long long>();
    init_block(nb, id_cap_);
    for (int a = 0; a < old_n_acc; ++a)
      AB_CUDA(cudaMemcpyAsync(nb + (size_t)a * id_cap_, old_blk + (size_t)a * id_cap_,
                              (size_t)n_valid * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, stream_));
    for (auto& pr : f64_from) {
      int grid = (int)std::min<uint64_t>((n_valid + 255) / 256 + 1, (uint64_t)num_sms_ * 8);
      i64_to_f64_kernel<<<grid, 256, 0, stream_>>>(old_blk + (size_t)pr.second * id_cap_, nb + (size_t)pr.first * id_cap_, n_valid);
      AB_CUDA(cudaGetLastError());
      ++st_.kernel_launches;
    }
    return nb;
  };
  for (auto& kv : panes_) {
    kv.second.dev = migrate(kv.second.dev);
    kv.second.frozen = migrate(kv.second.frozen);
    if (kv.second.slot >= 0) h_pane_ptrs_[kv.second.slot] = kv.second.dev;
  }
  for (auto& kv : zombies_) {
    kv.second.dev = migrate(kv.second.dev);
    kv.second.frozen = migrate(kv.second.frozen);
  }
  running_ = migrate(running_);
  AB_CUDA(cudaStreamSynchronize(stream_));
  free_panes_.clear();
  pane_storage_ = std::move(new_storage);
  ring_dirty_ = true;
}

// Leaves exact-sum AVG: every AVG gets its own f64 accumulator, seeded from the (still exact) integer sums.
void WindowAggOp::promote_avg() {
  if (!avg_exact_) return;
  AB_REQUIRE(in_flight_.empty(), ARROYO_B200_RUNTIME, "promote with launches in flight");
  const int old_n_acc = n_acc_;
  std::vector<std::pair<int, int>> f64_from;
  for (int g = 0; g < n_aggs_; ++g) {
    if (agg_kind_[g] != ARROYO_B200_AGG_AVG_I64) continue;
    const int src = agg_acc_[g];
    int found = -1;
    for (auto& pr : f64_from)
      if (pr.second == src) found = pr.first;
    if (found < 0) {
      AB_REQUIRE(n_acc_ < MAX_ACC, ARROYO_B200_RUNTIME, "too many accumulators after AVG promotion");
      found = n_acc_;
      acc_kind_[n_acc_] = ACC_SUM_F64;
      acc_val_[n_acc_] = acc_val_[src];
      ++n_acc_;
      f64_from.emplace_back(found, src);
    }
    agg_acc_[g] = found;
  }
  avg_exact_ = false;
  // f64 accumulators are not exactly invertible: leave running mode (see the constructor)
  if (running_mode_) {
    running_mode_ = false;
    in_running_.clear();
    for (auto& z : zombies_) {
      release_block(z.second.dev);
      release_block(z.second.frozen);
    }
    zombies_.clear();
    release_block(running_);
    running_ = nullptr;
  }
  relayout_blocks(old_n_acc, f64_from);
}

void WindowAggOp::ensure_pane(int64_t bin) {
  if (panes_.count(bin)) return;
  const uint64_t q = (uint64_t)bin / (uint64_t)slide_;
  while (true) {
    uint32_t slot = (uint32_t)q & (ring_ - 1);
    if (h_pane_bins_[slot] == FREE_BIN) break;
    // slot conflict: double the ring and re-place every live pane
    AB_REQUIRE(ring_ * 2 <= MAX_RING, ARROYO_B200_RUNTIME,
               "event-time spread of live panes exceeds the pane ring (4096 panes)");
    ring_ *= 2;
    std::fill(h_pane_bins_.begin(), h_pane_bins_.end(), FREE_BIN);
    std::fill(h_pane_ptrs_.begin(), h_pane_ptrs_.end(), nullptr);
    for (auto& kv : panes_) {
      if (kv.second.slot < 0) continue;
      uint32_t s = (uint32_t)((uint64_t)kv.first / (uint64_t)slide_) & (ring_ - 1);
      kv.second.slot = (int)s;
      h_pane_bins_[s] = kv.first;
      h_pane_ptrs_[s] = kv.second.dev;
    }
    ring_dirty_ = true;
  }
  Pane p;
  p.bin = bin;
  p.dev = acquire_block();
  p.slot = (int)((uint32_t)q & (ring_ - 1));
  h_pane_bins_[p.slot] = bin;
  h_pane_ptrs_[p.slot] = p.dev;
  panes_[bin] = p;
  ring_dirty_ = true;
}

void WindowAggOp::drop_pane(int64_t bin) {
  auto it = panes_.find(bin);
  if (it == panes_.end()) return;
  Pane& p = it->second;
  if (p.slot >= 0) {
    h_pane_bins_[p.slot] = FREE_BIN;
    h_pane_ptrs_[p.slot] = nullptr;
    ring_dirty_ = true;
  }
  release_block(p.dev);
  release_block(p.frozen);
  panes_.erase(it);
}

void WindowAggOp::upload_ring() {
  if (!ring_dirty_) return;
  // pageable sources: the runtime stages them before returning, so the vectors may change afterwards
  AB_CUDA(cudaMemcpyAsync(d_pane_bins_.p, h_pane_bins_.data(), ring_ * sizeof(long long), cudaMemcpyHostToDevice, stream_));
  AB_CUDA(cudaMemcpyAsync(d_pane_ptrs_.p, h_pane_ptrs_.data(), ring_ * sizeof(void*), cudaMemcpyHostToDevice, stream_));
  ring_dirty_ = false;
}

// Host->device copies of the input columns are submitted in groups with cudaMemcpyBatchAsync: a 64 Ki-row batch is
// three 512 KiB copies, and one cudaMemcpyAsync per copy tops out at 39 GB/s on this box's Gen5 x16 link where
// groups of 48 reach 55 GB/s (profiles/r01_pcie_probe2.txt) -- and cost a tenth of the host time.
void WindowAggOp::queue_copy(void* dst, const void* src, size_t bytes) {
  if (bytes == 0) return;
  copy_dst_.push_back(dst);
  copy_src_.push_back(const_cast<void*>(src));
  copy_size_.push_back(bytes);
  if (copy_dst_.size() >= COPY_GROUP) flush_copies();
}

void WindowAggOp::flush_copies() {
  const size_t n = copy_dst_.size();
  if (n == 0) return;
  bool done = false;
#if CUDART_VERSION >= 12080 && CUDART_VERSION < 13000  // CUDA 13 dropped the failIdx parameter
  if (batch_copy_ok_ && n > 1) {
    cudaMemcpyAttributes at{};
    at.srcAccessOrder = cudaMemcpySrcAccessOrderStream;  // the sources stay valid until the release event
    at.flags = cudaMemcpyFlagPreferOverlapWithCompute;
    size_t idx = 0, fail = 0;
    cudaError_t e = cudaMemcpyBatchAsync(copy_dst_.data(), copy_src_.data(), copy_size_.data(), n, &at, &idx, 1, &fail,
                                         copy_stream_);
    if (e == cudaSuccess) {
      done = true;
    } else if (e == cudaErrorNotSupported || e == cudaErrorInvalidValue) {
      cudaGetLastError();
      batch_copy_ok_ = false;  // e.g. pageable sources on a driver that refuses them: one copy at a time
    } else {
      AB_CUDA(e);
    }
  }
#endif
  if (!done)
    for (size_t i = 0; i < n; ++i)
      AB_CUDA(cudaMemcpyAsync(copy_dst_[i], copy_src_[i], copy_size_[i], cudaMemcpyHostToDevice, copy_stream_));
  copy_dst_.clear();
  copy_src_.clear();
  copy_size_.clear();
}

// Input batches are handed back in groups: one CUDA event per RELEASE_GROUP batches (or per launch / flush)
// instead of one per batch, and the events are recycled.
void WindowAggOp::seal_release() {
  flush_copies();
  if (open_release_.empty()) return;
  PendingRelease r;
  if (!ev_pool_.empty()) {
    r.ev = ev_pool_.back();
    ev_pool_.pop_back();
  } else {
    AB_CUDA(cudaEventCreateWithFlags(&r.ev, cudaEventDisableTiming));
  }
  AB_CUDA(cudaEventRecord(r.ev, copy_stream_));
  r.arrs.swap(open_release_);
  releases_.push_back(std::move(r));
}

void WindowAggOp::poll_releases(bool wait) {
  if (wait) seal_release();
  while (!releases_.empty()) {
    PendingRelease& r = releases_.front();
    if (wait) {
      AB_CUDA(cudaEventSynchronize(r.ev));
    } else {
      cudaError_t e = cudaEventQuery(r.ev);
      if (e == cudaErrorNotReady) break;
      AB_CUDA(e);
    }
    for (auto& a : r.arrs)
      if (a.release) a.release(&a);
    ev_pool_.push_back(r.ev);
    releases_.pop_front();
  }
}

void WindowAggOp::add_segment(const long long* key, const long long* ts, const long long* const* vals, int64_t n) {
  if (n <= 0) return;
  if (!segs_.empty()) {
    Segment& l = segs_.back();
    bool contig = l.ts + l.n == ts && (!keyed_ || l.key + l.n == key);
    for (int v = 0; v < n_vals_; ++v) contig = contig && (l.val[v] + l.n == vals[v]);
    if (contig) {
      l.n += n;
      pending_rows_ += n;
      return;
    }
  }
  if ((int)segs_.size() == MAX_SEGS) launch_pending();
  Segment s{};
  s.key = key;
  s.ts = ts;
  for (int v = 0; v < n_vals_; ++v) s.val[v] = vals[v];
  s.n = n;
  segs_.push_back(s);
  pending_rows_ += n;
}

void WindowAggOp::rotate_chunk() {
  cur_chunk_ = (cur_chunk_ + 1) % NCHUNK;
  cur_rows_ = 0;
  // the launch that last read this chunk must have finished before the copy engine writes it again (a wait on
  // the copy stream, not on the host)
  AB_CUDA(cudaStreamWaitEvent(copy_stream_, chunk_free_[cur_chunk_], 0));
}

void WindowAggOp::process_batch(uint32_t, uint32_t, ArrowArray* batch, const ArrowSchema* schema) {
  set_device();
  int64_t n = 0;
  std::vector<InColumn> cols = import_batch(batch, schema, &n);
  AB_REQUIRE((int)cols.size() == cfg.n_cols, ARROYO_B200_INVALID_ARGUMENT, "batch has the wrong number of columns");
  if (keyed_) key_format_ = cols[key_col_].format;
  for (int g = 0; g < n_aggs_; ++g)
    if (agg_kind_[g] == ARROYO_B200_AGG_MIN_I64 || agg_kind_[g] == ARROYO_B200_AGG_MAX_I64 ||
        agg_kind_[g] == ARROYO_B200_AGG_SUM_I64) {
      const std::string& f = cols[cfg.aggs[g].input_col].format;
      AB_REQUIRE(f != "g", ARROYO_B200_UNSUPPORTED, "float64 aggregate inputs are not supported");
      if (agg_kind_[g] != ARROYO_B200_AGG_SUM_I64) agg_format_[g] = f;
    }
  poll_releases(false);
  st_.rows_in += (uint64_t)n;
  if (n > 0 && panes_.empty() && max_bin_seen_ == LLONG_MIN) {
    // residency hint only (no semantics): make the first row's pane resident so a cold start does
    // not have to go through the deferred path
    int64_t b0 = bin_start((int64_t)cols[ts_col_].data[0], slide_);
    if (b0 >= late_bin_) {
      ensure_pane(b0);
      max_bin_seen_ = b0;
      lookahead();
    }
  }
  // ARROYO_B200_FLAG_ZERO_COPY: pinned (page-locked, device-mapped) Arrow buffers are read in place by the
  // ingest kernel over PCIe: no staging memory.  Measured slower than DMA staging on this pool's hosts
  // (0.96 vs 1.22 G rows/s end to end: SM loads over PCIe ~23 GB/s vs copy engine ~29 GB/s), hence opt-in.
  if (n > 0 && (cfg.flags & ARROYO_B200_FLAG_ZERO_COPY)) {
    bool pinned = true;
    const uint64_t* devp[ARROYO_B200_MAX_COLS] = {nullptr};
    auto probe = [&](int c) {
      cudaPointerAttributes at{};
      if (cudaPointerGetAttributes(&at, cols[c].data) != cudaSuccess) {
        cudaGetLastError();
        pinned = false;
        return;
      }
      if (at.type != cudaMemoryTypeHost || at.devicePointer == nullptr) pinned = false;
      else devp[c] = (const uint64_t*)at.devicePointer;
    };
    if (keyed_) probe(key_col_);
    probe(ts_col_);
    for (int v = 0; v < n_vals_; ++v) probe(val_cols_[v]);
    if (pinned) {
      int64_t done = 0;
      while (done < n) {
        int64_t take = std::min<int64_t>(n - done, launch_rows_ - pending_rows_);
        const long long* vals[MAX_VALS];
        for (int v = 0; v < n_vals_; ++v) vals[v] = (const long long*)devp[val_cols_[v]] + done;
        add_segment(keyed_ ? (const long long*)devp[key_col_] + done : nullptr, (const long long*)devp[ts_col_] + done,
                    vals, take);
        done += take;
        if (done < n && pending_rows_ >= launch_rows_) launch_pending();
      }
      st_.h2d_bytes += (uint64_t)n * 8 * (uint64_t)((keyed_ ? 1 : 0) + 1 + n_vals_);
      zero_copy_inputs_.push_back(*batch);
      batch->release = nullptr;
      if (pending_rows_ >= launch_rows_) launch_pending();
      return;
    }
  }
  const int n_used = 2 + n_vals_;
  int64_t done = 0;
  while (done < n) {
    if (!chunk_[cur_chunk_].p) chunk_[cur_chunk_].alloc((size_t)n_used * chunk_rows_ * 8);
    int64_t room = chunk_rows_ - cur_rows_;
    if (room == 0) {
      launch_pending();
      rotate_chunk();
      continue;
    }
    int64_t take = std::min(room, n - done);
    long long* base = chunk_[cur_chunk_].as<long long>();
    long long* d_key = base + 0 * chunk_rows_ + cur_rows_;
    long long* d_ts = base + 1 * chunk_rows_ + cur_rows_;
    const long long* d_vals[MAX_VALS];
    if (keyed_) queue_copy(d_key, cols[key_col_].data + done, (size_t)take * 8);
    queue_copy(d_ts, cols[ts_col_].data + done, (size_t)take * 8);
    for (int v = 0; v < n_vals_; ++v) {
      long long* dv = base + (size_t)(2 + v) * chunk_rows_ + cur_rows_;
      queue_copy(dv, cols[val_cols_[v]].data + done, (size_t)take * 8);
      d_vals[v] = dv;
    }
    st_.h2d_bytes += (uint64_t)take * 8 * (uint64_t)((keyed_ ? 1 : 0) + 1 + n_vals_);
    add_segment(d_key, d_ts, d_vals, take);
    pending_uses_chunk_ = true;
    cur_rows_ += take;
    done += take;
  }
  // ownership of the input moves to the library; released once the copies have completed
  open_release_.push_back(*batch);
  batch->release = nullptr;
  if (open_release_.size() >= RELEASE_GROUP) seal_release();
  if (cur_rows_ == chunk_rows_) {
    launch_pending();
    rotate_chunk();
  }
}

void WindowAggOp::process_device_batch(uint32_t, uint32_t, const uint64_t* cols, int32_t n_cols, int64_t n_rows) {
  set_device();
  AB_REQUIRE(n_cols == cfg.n_cols, ARROYO_B200_INVALID_ARGUMENT, "batch has the wrong number of columns");
  if (n_rows <= 0) return;
  st_.rows_in += (uint64_t)n_rows;
  int64_t done = 0;
  while (done < n_rows) {
    int64_t take = std::min<int64_t>(n_rows - done, launch_rows_ - pending_rows_);
    const long long* vals[MAX_VALS];
    for (int v = 0; v < n_vals_; ++v) vals[v] = (const long long*)cols[val_cols_[v]] + done;
    add_segment(keyed_ ? (const long long*)cols[key_col_] + done : nullptr, (const long long*)cols[ts_col_] + done, vals,
                take);
    done += take;
    if (pending_rows_ >= launch_rows_) launch_pending();
  }
}

// The two-pass ingest handles the plans whose accumulators are {rows} or {rows, wrapping SUM(Int64) of one column}
// over raw input rows (COUNT(*), SUM, AVG-from-exact-sum: the headline), when the launch is large enough to pay for
// the per-bucket set-up and the dictionary fits the partition kernel's histograms.  Everything else -- and every row
// the two passes hand back -- runs through the one-pass kernel.
bool WindowAggOp::two_pass_eligible(uint64_t rows) const {
  if (!two_pass_enabled_ || !keyed_ || rows_slot_ >= 0 || n_vals_ > 1 || n_acc_ > 2) return false;
  if (n_acc_ == 2 && acc_kind_[1] != ACC_SUM_I64) return false;
  if (n_buckets_ > (uint64_t)P1_NR) return false;
  if (max_bin_seen_ == LLONG_MIN) return false;  // no pane known yet: the first launch finds out where the stream is
  if (two_pass_pause_ > 0) {
    --two_pass_pause_;
    return false;
  }
  static const uint64_t min_rows = [] {
    const char* e = getenv("ARROYO_B200_TWO_PASS_MIN_ROWS");
    return e ? strtoull(e, nullptr, 10) : (1ull << 19);
  }();
  return rows >= min_rows || (cfg.flags & ARROYO_B200_FLAG_TWO_PASS_ALWAYS);
}

void WindowAggOp::launch_two_pass(IngestParams& p, uint64_t rows, long long tiles) {
  TwoPassParams tp{};
  // fast panes: the newest pane seen and the next one (in-order streams write nothing else)
  int nf = 0;
  for (int k = 0; k < 3 && nf < TP_NP; ++k) {
    const int64_t b = max_bin_seen_ + (int64_t)(k == 2 ? -1 : k) * slide_;
    auto it = panes_.find(b);
    if (b < late_bin_ || it == panes_.end() || it->second.slot < 0) continue;
    tp.fast_q[nf] = (unsigned long long)b / (unsigned long long)slide_;
    tp.fast_ptr[nf] = it->second.dev;
    tp.fast_slot[nf] = (uint32_t)it->second.slot;
    ++nf;
  }
  for (int f = nf; f < TP_NP; ++f) {
    tp.fast_q[f] = ~0ull;
    tp.fast_ptr[f] = nullptr;
    tp.fast_slot[f] = 0;
  }
  const uint32_t n_regions = (uint32_t)(TP_NP * n_buckets_);
  // a region holds a bucket's share of one pane's rows: mean rows / buckets, plus slack for the spread
  const uint64_t mean = (uint64_t)launch_rows_ / n_buckets_ + 1;
  const uint32_t cap = (uint32_t)std::min<uint64_t>(((mean + mean / 4 + 2048 + 63) / 64) * 64, 1u << 30);
  if (part_cap_ != cap || !part_.p) {
    AB_CUDA(cudaStreamSynchronize(stream_));
    part_.alloc((size_t)n_regions * cap * sizeof(Rec));
    part_cursor_.alloc((size_t)2 * n_regions * sizeof(unsigned int));
    AB_CUDA(cudaMemsetAsync(part_cursor_.p, 0, (size_t)2 * n_regions * sizeof(unsigned int), stream_));
    part_cap_ = cap;
  }
  tp.part = part_.as<Rec>();
  tp.cursor = part_cursor_.as<unsigned int>() + (size_t)part_flip_ * n_regions;
  tp.cursor_next = part_cursor_.as<unsigned int>() + (size_t)(part_flip_ ^ 1) * n_regions;
  part_flip_ ^= 1;
  tp.cap = cap;
  // blocks per region in pass 2: enough blocks to fill the GPU when there are few buckets
  const uint32_t want_blocks = (uint32_t)num_sms_ * 2;
  tp.slices = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((want_blocks + n_buckets_ - 1) / n_buckets_,
                                                                 std::max<uint64_t>(1, rows / n_buckets_ / 4096)));
  if (!two_pass_attr_set_) {
    AB_CUDA(cudaFuncSetAttribute(part_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P1_SMEM));
    AB_CUDA(cudaFuncSetAttribute(part_kernel<1, sig_of(ACC_SUM_I64)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P1_SMEM));
    AB_CUDA(cudaFuncSetAttribute(agg_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2_SMEM));
    AB_CUDA(cudaFuncSetAttribute(agg_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2_SMEM));
    two_pass_attr_set_ = true;
  }
  const int grid1 = (int)std::max<long long>(1, std::min<long long>(tiles, (long long)num_sms_ * P1_BLOCKS_PER_SM));
  // Blocks take work items round-robin.  With one item per bucket the last round is ragged (1024 buckets over 296
  // blocks: the fourth round keeps 136 blocks busy and 160 idle for a whole bucket); cutting the buckets of that round
  // into slices turns it into a short round of part-buckets (each slice builds the bucket's table again).
  const uint32_t max_blocks = (uint32_t)num_sms_ * P2_BLOCKS_PER_SM;
  tp.tail_first = (uint32_t)n_buckets_;
  tp.tail_slices = 1;
  if (tp.slices == 1 && n_buckets_ > max_blocks && rows / n_buckets_ >= 2048) {
    const uint32_t rest = (uint32_t)(n_buckets_ % max_blocks);
    if (rest && max_blocks / rest >= 2) {
      tp.tail_first = (uint32_t)n_buckets_ - rest;
      tp.tail_slices = std::min<uint32_t>(max_blocks / rest, 4);
    }
  }
  const uint32_t n_work = tp.tail_first * tp.slices + ((uint32_t)n_buckets_ - tp.tail_first) * tp.tail_slices;
  const int grid2 = (int)std::max<uint32_t>(1, std::min<uint32_t>(n_work, max_blocks));
  if (n_vals_ == 0) {
    part_kernel<0, 0><<<grid1, P1_THREADS, P1_SMEM, stream_>>>(p, tp);
    AB_CUDA(cudaGetLastError());
    agg_kernel<0><<<grid2, P2_NW * 32, P2_SMEM, stream_>>>(p, tp);
  } else {
    part_kernel<1, sig_of(ACC_SUM_I64)><<<grid1, P1_THREADS, P1_SMEM, stream_>>>(p, tp);
    AB_CUDA(cudaGetLastError());
    agg_kernel<1><<<grid2, P2_NW * 32, P2_SMEM, stream_>>>(p, tp);
  }
  ++st_.kernel_launches;  // (the second kernel is counted by the caller)
}

void WindowAggOp::launch_segments(const std::vector<Segment>& segs_in, int chunk) {
  // At most two launches (each <= launch_rows_ rows) are ever in flight, so the deferred buffer
  // (2 * launch_rows_ rows) cannot overflow; as soon as a finished launch reports deferrals they are
  // drained before anything else is queued.
  while (in_flight_.size() >= 2) absorb(in_flight_.front());
  if (!draining_ && have_counters_ && last_counters_.deferred > 0) {
    while (!in_flight_.empty()) absorb(in_flight_.front());
    drain_deferred();
  }
  const int li = next_launch_;
  next_launch_ = (next_launch_ + 1) % NLAUNCH;
  LaunchRec& L = launches_[li];
  AB_REQUIRE(!L.in_flight, ARROYO_B200_RUNTIME, "launch record still in flight");
  Segment* hs = h_segs_[li].as<Segment>();
  long long tiles = 0;
  uint64_t rows = 0;
  for (size_t i = 0; i < segs_in.size(); ++i) {
    hs[i] = segs_in[i];
    hs[i].tile_start = tiles;
    uintptr_t al = (uintptr_t)hs[i].ts;
    if (keyed_) al |= (uintptr_t)hs[i].key;
    for (int v = 0; v < n_vals_; ++v) al |= (uintptr_t)hs[i].val[v];
    hs[i].vec_ok = (al & 15) == 0;
    tiles += (hs[i].n + TILE - 1) / TILE;
    rows += (uint64_t)hs[i].n;
  }
  const bool two_pass = two_pass_eligible(rows);
  long long t2 = 0;
  if (two_pass) {
    // tiles of the partition kernel are larger: the segment table is cut for them
    for (size_t i = 0; i < segs_in.size(); ++i) {
      hs[i].tile_start = t2;
      t2 += (hs[i].n + P1_TILE - 1) / P1_TILE;
    }
  }
  AB_CUDA(cudaMemcpyAsync(d_segs_[li].p, hs, segs_in.size() * sizeof(Segment), cudaMemcpyHostToDevice, stream_));
  if (ring_ > RING_INLINE) upload_ring();
  if (!defer_[defer_cur_][0].p) {
    for (int c = 0; c < 2 + n_vals_; ++c) defer_[defer_cur_][c].alloc(defer_cap_ * 8);
  }

  IngestParams p{};
  p.segs = d_segs_[li].as<Segment>();
  p.n_segs = (int)segs_in.size();
  p.keyed = keyed_ ? 1 : 0;
  p.n_tiles = tiles;
  p.dict = dict_view();
  p.slide_div = FastDivU64::make((uint64_t)slide_);
  p.slide = slide_;
  p.late_bin = late_bin_;
  p.late_q = late_bin_ == LLONG_MIN ? 0ull : (unsigned long long)late_bin_ / (unsigned long long)slide_;
  p.guard_vals = avg_exact_ ? guard_vals_ : 0u;
  p.combine = (cfg.flags & ARROYO_B200_FLAG_NO_COMBINE) ? 0 : 1;
  p.rows_slot = rows_slot_;
  p.ring_mask = ring_ - 1;
  p.n_acc = n_acc_;
  p.pane_bins = d_pane_bins_.as<long long>();
  p.pane_ptrs = d_pane_ptrs_.as<unsigned long long*>();
  p.id_cap = id_cap_;
  p.ring_inline = ring_ <= RING_INLINE ? 1 : 0;
  if (p.ring_inline)
    for (uint32_t i = 0; i < ring_; ++i) {
      p.ring_bins[i] = h_pane_bins_[i];
      p.ring_ptrs[i] = h_pane_ptrs_[i];
    }
  for (int a = 0; a < n_acc_; ++a) {
    p.acc_kind[a] = acc_kind_[a];
    p.acc_val[a] = acc_val_[a];
  }
  p.counters = d_counters();
  p.slot_rows = d_slot_rows();
  p.d_key = defer_[defer_cur_][0].as<long long>();
  p.d_ts = defer_[defer_cur_][1].as<long long>();
  for (int v = 0; v < n_vals_; ++v) p.d_val[v] = defer_[defer_cur_][2 + v].as<long long>();
  p.defer_cap = defer_cap_;

  int grid = (int)std::min<long long>(tiles, (long long)num_sms_ * 8);
  if (grid < 1) grid = 1;
  if (profile_) AB_CUDA(cudaEventRecord(L.t0, stream_));
  if (two_pass) {
    p.n_tiles = t2;
    launch_two_pass(p, rows, t2);
  }
  // straight-line specialisations for the common accumulator signatures, generic otherwise
  int sig = GENERIC_SIG;
  if (n_vals_ <= 1 && n_acc_ <= 4) {
    int k[3] = {0, 0, 0};
    for (int a = 1; a < n_acc_; ++a) k[a - 1] = acc_kind_[a];
    sig = sig_of(k[0], k[1], k[2]);
  }
#define AB_LAUNCH(NV, SIG) ingest_kernel<NV, SIG><<<grid, THREADS, 0, stream_>>>(p)
  if (two_pass) {
    // launched above
  } else if (n_vals_ == 0) AB_LAUNCH(0, 0);
  else if (n_vals_ == 1 && sig == sig_of(ACC_SUM_I64)) AB_LAUNCH(1, sig_of(ACC_SUM_I64));
  else if (n_vals_ == 1 && sig == sig_of(ACC_SUM_F64)) AB_LAUNCH(1, sig_of(ACC_SUM_F64));
  else if (n_vals_ == 1 && sig == sig_of(ACC_SUM_I64, ACC_SUM_F64)) AB_LAUNCH(1, sig_of(ACC_SUM_I64, ACC_SUM_F64));
  else if (n_vals_ == 1 && sig == sig_of(ACC_MIN_I64, ACC_MAX_I64)) AB_LAUNCH(1, sig_of(ACC_MIN_I64, ACC_MAX_I64));
  else if (n_vals_ == 1) AB_LAUNCH(1, GENERIC_SIG);
  else if (n_vals_ == 2) AB_LAUNCH(2, GENERIC_SIG);
  else if (n_vals_ == 3) AB_LAUNCH(3, GENERIC_SIG);
  else AB_LAUNCH(4, GENERIC_SIG);
#undef AB_LAUNCH
  AB_CUDA(cudaGetLastError());
  if (profile_) AB_CUDA(cudaEventRecord(L.t1, stream_));
  ++st_.kernel_launches;
  ++st_.ingest_launches;
  AB_CUDA(cudaMemcpyAsync(L.h_counters, book_.p, BOOK_SLOT_OFF + ring_ * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                          stream_));
  AB_CUDA(cudaEventRecord(L.done, stream_));
  if (chunk >= 0) AB_CUDA(cudaEventRecord(chunk_free_[chunk], stream_));
  L.rows = rows;
  L.in_flight = true;
  L.chunk = chunk;
  in_flight_.push_back(li);
}

void WindowAggOp::launch_pending() {
  seal_release();
  if (segs_.empty()) return;
  std::vector<Segment> segs;
  segs.swap(segs_);
  pending_rows_ = 0;
  int chunk = pending_uses_chunk_ ? cur_chunk_ : -1;
  pending_uses_chunk_ = false;
  if (chunk >= 0) {
    // the kernel reads staged rows: it runs behind the copies that were queued up to here
    AB_CUDA(cudaEventRecord(copied_, copy_stream_));
    AB_CUDA(cudaStreamWaitEvent(stream_, copied_, 0));
  }
  launch_segments(segs, chunk);
  if (!zero_copy_inputs_.empty()) {
    // the pinned input batches these segments point into may be released once this kernel has run
    PendingRelease r;
    if (!ev_pool_.empty()) {
      r.ev = ev_pool_.back();
      ev_pool_.pop_back();
    } else {
      AB_CUDA(cudaEventCreateWithFlags(&r.ev, cudaEventDisableTiming));
    }
    AB_CUDA(cudaEventRecord(r.ev, stream_));
    r.arrs.swap(zero_copy_inputs_);
    releases_.push_back(std::move(r));
  }
}

void WindowAggOp::touch(int64_t bin) {
  if (sliding_) sliding_planner_->touch(bin);
  else tumbling_->touch(bin);
}

// Waits for one launch and folds its bookkeeping into the host state machine.
void WindowAggOp::absorb(int li) {
  LaunchRec& L = launches_[li];
  AB_REQUIRE(L.in_flight, ARROYO_B200_RUNTIME, "absorb of an idle launch");
  AB_CUDA(cudaEventSynchronize(L.done));
  L.in_flight = false;
  AB_REQUIRE(!in_flight_.empty() && in_flight_.front() == li, ARROYO_B200_RUNTIME, "launch order violated");
  in_flight_.pop_front();
  if (profile_) {
    float ms = 0;
    AB_CUDA(cudaEventElapsedTime(&ms, L.t0, L.t1));
    st_.ingest_ms += ms;
    st_.ingest_rows_timed += L.rows;
  }
  const Counters& c = *L.h_counters;
  last_counters_ = c;
  have_counters_ = true;
  total_keys_host_ = c.n_keys;
  if (c.part_overflow != part_overflow_seen_) {
    // a launch whose rows pile up in a few buckets (a hot key) is the one-pass kernel's case: its warp-combine turns
    // the hot key's rows into one update per warp.  Skewed streams stay skewed: the two-pass path is retried later.
    if (c.part_overflow - part_overflow_seen_ > L.rows / 64) two_pass_pause_ = 64;
    part_overflow_seen_ = c.part_overflow;
  }
  if (c.max_q) max_bin_seen_ = std::max<int64_t>(max_bin_seen_, (int64_t)(c.max_q * (uint64_t)slide_));
  for (uint32_t s = 0; s < ring_; ++s) {
    const unsigned long long fresh = L.h_slot_rows[s] - slot_rows_seen_[s];  // cumulative on the device
    slot_rows_seen_[s] = L.h_slot_rows[s];
    if (fresh) {
      AB_REQUIRE(h_pane_bins_[s] != FREE_BIN, ARROYO_B200_RUNTIME, "touched a free ring slot");
      Pane& tp = panes_.at(h_pane_bins_[s]);
      tp.rows += fresh;
      if (tp.rows >= (1ull << 31)) need_promote_ = true;
      touch(h_pane_bins_[s]);
    }
  }
  if (c.lost) throw Error(ARROYO_B200_RUNTIME, "deferred-row buffer overflowed; rows were lost");
  if (c.neg_ts)
    throw Error(ARROYO_B200_PANIC, "batch holds a negative _timestamp (before the Unix epoch): the reference panics on it");
  lookahead();
}

// Keep panes resident a little ahead of the newest bin seen so in-order streams never defer.
void WindowAggOp::lookahead() {
  if (max_bin_seen_ == LLONG_MIN) return;
  for (int k = 0; k <= 2; ++k) {
    int64_t b = max_bin_seen_ + (int64_t)k * slide_;
    if (b >= late_bin_ && !panes_.count(b)) {
      // only if the slot is free: never grow the ring speculatively
      uint32_t slot = (uint32_t)((uint64_t)b / (uint64_t)slide_) & (ring_ - 1);
      if (h_pane_bins_[slot] == FREE_BIN) ensure_pane(b);
    }
  }
}

void WindowAggOp::sync_all() {
  while (!in_flight_.empty()) absorb(in_flight_.front());
  if (need_promote_ && avg_exact_) promote_avg();
  drain_deferred();
}

// Slow path: rows the kernel could not place (pane not resident, dictionary full).  Grows what is
// missing and re-ingests them; loops until nothing is deferred.
void WindowAggOp::drain_deferred() {
  struct Guard {
    bool& f;
    explicit Guard(bool& x) : f(x) { f = true; }
    ~Guard() { f = false; }
  } guard(draining_);
  for (int iter = 0; iter < 64; ++iter) {
    if (!have_counters_ || last_counters_.deferred == 0) return;
    AB_REQUIRE(in_flight_.empty(), ARROYO_B200_RUNTIME, "drain with launches in flight");
    const uint64_t n = last_counters_.deferred;
    AB_REQUIRE(n <= defer_cap_, ARROYO_B200_RUNTIME, "deferred overflow");
    st_.rows_deferred += n;
    // which panes do the deferred rows need?
    std::vector<long long> ts(n);
    AB_CUDA(cudaMemcpyAsync(ts.data(), defer_[defer_cur_][1].p, n * 8, cudaMemcpyDeviceToHost, stream_));
    AB_CUDA(cudaStreamSynchronize(stream_));
    std::set<int64_t> bins;
    for (uint64_t i = 0; i < n; ++i) {
      int64_t b = (int64_t)((uint64_t)ts[i] / (uint64_t)slide_ * (uint64_t)slide_);
      if (b >= late_bin_) bins.insert(b);
    }
    for (int64_t b : bins) ensure_pane(b);
    if (last_counters_.big_vals && avg_exact_) promote_avg();
    // dictionary pressure: a bucket ran out of ids (its rows were deferred), or the mean bucket fill is past the
    // point where that becomes likely: double the bucket count
    if (keyed_ && (last_counters_.dict_full != dict_full_seen_ ||
                   (uint64_t)last_counters_.n_keys > n_buckets_ * (uint64_t)(BD_MEAN + BD_MEAN / 8))) {
      dict_full_seen_ = last_counters_.dict_full;
      grow_ids();
      last_counters_.n_keys = total_keys_host_;
    }
    // re-ingest from the filled set while new deferrals go to the other set
    const int full = defer_cur_;
    defer_cur_ ^= 1;
    unsigned long long zero = 0;
    AB_CUDA(cudaMemcpyAsync((char*)book_.p + offsetof(Counters, deferred), &zero, sizeof zero,
                            cudaMemcpyHostToDevice, stream_));
    Segment s{};
    s.key = defer_[full][0].as<long long>();
    s.ts = defer_[full][1].as<long long>();
    for (int v = 0; v < n_vals_; ++v) s.val[v] = defer_[full][2 + v].as<long long>();
    s.n = (long long)n;
    // deferred rows were already counted (late rows among them are counted when re-ingested)
    launch_segments({s}, -1);
    while (!in_flight_.empty()) absorb(in_flight_.front());
  }
  throw Error(ARROYO_B200_RUNTIME, "deferred rows did not converge");
}

void WindowAggOp::flush() {
  set_device();
  resolve_deferred();
  launch_pending();
  sync_all();
  poll_releases(true);
}

void WindowAggOp::submit() {
  set_device();
  launch_pending();
}

// The output buffers of the previous emission may still be in flight to the host.
void WindowAggOp::wait_outputs() {
  if (!out_inflight_) return;
  AB_CUDA(cudaEventSynchronize(out_done_));
  out_inflight_ = false;
}

void WindowAggOp::begin_watermark(int64_t wm) {
  set_device();
  if (!out_stream_) {
    AB_CUDA(cudaStreamCreateWithFlags(&out_stream_, cudaStreamNonBlocking));
    AB_CUDA(cudaEventCreateWithFlags(&emit_done_, cudaEventDisableTiming));
    AB_CUDA(cudaEventCreateWithFlags(&out_done_, cudaEventDisableTiming));
  }
  struct Flag {
    bool& f;
    explicit Flag(bool& x) : f(x) { f = true; }
    ~Flag() { f = false; }
  } flag(async_out_);
  handle_watermark(wm, pending_out, nullptr);
  AB_CUDA(cudaEventRecord(out_done_, out_stream_));
  out_inflight_ = true;
}

bool WindowAggOp::poll_watermark(bool block) {
  if (!out_inflight_) return true;
  set_device();
  if (block) {
    wait_outputs();
    return true;
  }
  cudaError_t e = cudaEventQuery(out_done_);
  if (e == cudaErrorNotReady) return false;
  AB_CUDA(e);
  out_inflight_ = false;
  return true;
}

WindowAggOp::OutSet* WindowAggOp::out_set(size_t i, uint64_t cap) {
  while (out_sets_.size() <= i) out_sets_.emplace_back(new OutSet());
  OutSet* os = out_sets_[i].get();
  if (os->cap < cap) {
    uint64_t c = std::max<uint64_t>(std::max<uint64_t>(cap, id_cap_), 1024);
    os->key.alloc(c * 8);
    os->wstart.alloc(c * 8);
    os->wend.alloc(c * 8);
    os->ts.alloc(c * 8);
    for (int g = 0; g < n_aggs_; ++g) os->agg[g].alloc(c * 8);
    os->cap = c;
    for (int a = 0; a < MAX_ACC; ++a) os->state[a].release();
  }
  return os;
}

// Runs the merge/emit kernel; returns the number of output rows (synchronises on the count).
int64_t WindowAggOp::run_emit(const std::vector<const unsigned long long*>& blocks, int n_add, bool use_running,
                              bool partial, int64_t wstart, int64_t wend, int64_t ts, OutSet* os) {
  AB_REQUIRE(blocks.size() <= (size_t)MAX_MERGE, ARROYO_B200_RUNTIME, "too many panes in one window");
  const uint32_t n_ids = n_keys_host_;
  EmitParams p{};
  p.panes_inline = blocks.size() <= (size_t)EMIT_INLINE ? 1 : 0;
  if (p.panes_inline) {
    for (size_t i = 0; i < blocks.size(); ++i) p.inline_panes[i] = blocks[i];
  } else {
    AB_CUDA(cudaMemcpyAsync(d_emit_panes_.p, blocks.data(), blocks.size() * sizeof(void*), cudaMemcpyHostToDevice, stream_));
  }
  p.panes = d_emit_panes_.as<const unsigned long long*>();
  p.n_panes = (int)blocks.size();
  p.n_acc = n_acc_;
  p.id_cap = id_cap_;
  p.n_ids = n_ids;
  p.keyed = keyed_ ? 1 : 0;
  for (int a = 0; a < n_acc_; ++a) p.acc_kind[a] = acc_kind_[a];
  std::vector<std::pair<unsigned long long*, unsigned long long*>> dup_cols;  // (src, dst): same output twice
  for (int a = 0; a < MAX_ACC; ++a) {
    p.out_raw[a] = nullptr;
    p.out_avg[a] = nullptr;
  }
  if (!partial) {
    for (int g = 0; g < n_aggs_; ++g) {
      unsigned long long* col = os->agg[g].as<unsigned long long>();
      const bool avg = agg_kind_[g] == ARROYO_B200_AGG_AVG_I64;
      const int a = agg_kind_[g] == ARROYO_B200_AGG_COUNT_STAR ? 0 : agg_acc_[g];
      unsigned long long*& slot = avg ? p.out_avg[a] : p.out_raw[a];
      if (slot) dup_cols.emplace_back(slot, col);
      else slot = col;
    }
  }
  p.id_keys = id_keys_.as<long long>();
  p.out_key = os->key.as<long long>();
  const bool proj = cfg.final_projection != 0 && !partial;
  p.out_wstart = proj ? os->wstart.as<long long>() : nullptr;
  p.out_wend = proj ? os->wend.as<long long>() : nullptr;
  p.out_ts = os->ts.as<long long>();
  p.wstart = wstart;
  p.wend = wend;
  p.ts = ts;
  p.out_count = d_out_count_.as<unsigned int>();
  const bool deferred = defer_counts_ && count_slots_used_ < COUNT_SLOTS;
  if (defer_counts_) {
    // nobody on the host knows the counter's value before the previous window's count has come back: restart it
    AB_CUDA(cudaMemsetAsync(d_out_count_.p, 0, sizeof(unsigned int), stream_));
    out_count_base_ = 0;
  }
  p.out_base = out_count_base_;
  p.running = use_running ? running_ : nullptr;
  p.n_add = n_add;
  p.partial = partial ? 1 : 0;
  if (partial) {
    for (int a = 0; a < n_acc_; ++a) {
      if (!os->state[a].p) os->state[a].alloc(os->cap * 8);
      p.out_state[a] = os->state[a].as<unsigned long long>();
    }
  }
  const uint32_t n_iter = ((n_ids + 1) / 2 + EMIT_THREADS - 1) / EMIT_THREADS;
  int grid = (int)std::min<uint32_t>(std::max<uint32_t>(n_iter, 1u), (uint32_t)num_sms_ * 8);
  if (profile_) {
    if (emit_events_used_ == emit_events_.size()) {
      cudaEvent_t e0 = nullptr, e1 = nullptr;
      AB_CUDA(cudaEventCreate(&e0));
      AB_CUDA(cudaEventCreate(&e1));
      emit_events_.emplace_back(e0, e1);
    }
    AB_CUDA(cudaEventRecord(emit_events_[emit_events_used_].first, stream_));
  }
#define AB_EMIT(N)                                                               \
  do {                                                                          \
    if (use_running) emit_kernel<true, N><<<grid, EMIT_THREADS, 0, stream_>>>(p); \
    else emit_kernel<false, N><<<grid, EMIT_THREADS, 0, stream_>>>(p);            \
  } while (0)
  switch (n_acc_) {
    case 1: AB_EMIT(1); break;
    case 2: AB_EMIT(2); break;
    case 3: AB_EMIT(3); break;
    case 4: AB_EMIT(4); break;
    case 5: AB_EMIT(5); break;
    case 6: AB_EMIT(6); break;
    case 7: AB_EMIT(7); break;
    case 8: AB_EMIT(8); break;
    default: AB_EMIT(9); break;
  }
  static_assert(MAX_ACC == 9, "emit_kernel instantiations cover 1..MAX_ACC accumulators");
#undef AB_EMIT
  AB_CUDA(cudaGetLastError());
  if (profile_) {
    AB_CUDA(cudaEventRecord(emit_events_[emit_events_used_].second, stream_));
    ++emit_events_used_;
    st_.emit_rows_timed += n_ids;
  }
  ++st_.kernel_launches;
  ++st_.emit_launches;
  if (deferred) {
    const int slot = count_slots_used_++;
    AB_CUDA(cudaMemcpyAsync(h_out_counts_.as<unsigned int>() + slot, d_out_count_.p, sizeof(unsigned int),
                            cudaMemcpyDeviceToHost, stream_));
    counts_pending_ = true;
    for (auto& d : dup_cols)  // row count unknown here: every id's worth
      if (n_ids) AB_CUDA(cudaMemcpyAsync(d.second, d.first, (size_t)n_ids * 8, cudaMemcpyDeviceToDevice, stream_));
    return -(int64_t)(slot + 1);
  }
  AB_CUDA(cudaMemcpyAsync(h_out_count_.p, d_out_count_.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, stream_));
  AB_CUDA(cudaStreamSynchronize(stream_));
  const unsigned int out_now = *h_out_count_.as<unsigned int>();
  const int64_t n_out = (int64_t)(unsigned int)(out_now - out_count_base_);
  out_count_base_ = out_now;
  for (auto& d : dup_cols)
    if (n_out) AB_CUDA(cudaMemcpyAsync(d.second, d.first, (size_t)n_out * 8, cudaMemcpyDeviceToDevice, stream_));
  return n_out;
}

static void* d2h_column(const void* dev, int64_t n, cudaStream_t s, uint64_t* bytes) {
  void* h = PinnedPool::get().alloc((size_t)std::max<int64_t>(n, 1) * 8);
  if (n > 0) AB_CUDA(cudaMemcpyAsync(h, dev, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
  *bytes += (uint64_t)n * 8;
  return h;
}

// Output batch in the operator's out_schema order: aggregate output columns [key?, aggs...] with the
// window struct inserted at window_index, then _timestamp (planner extension/aggregate.rs:306-389).
void WindowAggOp::export_window(OutSet* os, int64_t n, BatchesPriv* out_host) {
  cudaStream_t cs = stream_;
  if (async_out_) {
    // the copies run behind everything the emission enqueued on the compute stream
    AB_CUDA(cudaEventRecord(emit_done_, stream_));
    AB_CUDA(cudaStreamWaitEvent(out_stream_, emit_done_, 0));
    cs = out_stream_;
  }
  std::vector<OutColumn> cols;
  if (keyed_) {
    OutColumn k;
    k.name = "key";
    k.format = key_format_;
    k.data = d2h_column(os->key.p, n, cs, &st_.d2h_bytes);
    cols.push_back(k);
  }
  for (int g = 0; g < n_aggs_; ++g) {
    OutColumn a;
    a.name = "agg" + std::to_string(g);
    a.format = agg_format_[g];
    a.data = d2h_column(os->agg[g].p, n, cs, &st_.d2h_bytes);
    cols.push_back(a);
  }
  if (cfg.final_projection) {
    OutColumn w;
    w.name = "window";
    w.format = "+s";
    OutColumn ws, we;
    ws.name = "start";
    ws.format = "tsn:";
    ws.data = d2h_column(os->wstart.p, n, cs, &st_.d2h_bytes);
    we.name = "end";
    we.format = "tsn:";
    we.data = d2h_column(os->wend.p, n, cs, &st_.d2h_bytes);
    w.children = {ws, we};
    int wi = std::min<int>(std::max<int>(cfg.window_index, 0), (int)cols.size());
    cols.insert(cols.begin() + wi, w);
  }
  OutColumn t;
  t.name = "_timestamp";
  t.format = "tsn:";
  t.data = d2h_column(os->ts.p, n, cs, &st_.d2h_bytes);
  cols.push_back(t);
  if (!async_out_) AB_CUDA(cudaStreamSynchronize(stream_));
  out_host->arrays.emplace_back();
  out_host->schemas.emplace_back();
  export_batch(cols, n, &out_host->arrays.back(), &out_host->schemas.back());
}

// Partial-state batch in `partial_schema`: [key?, state cols..., _timestamp = pane start]
// (arroyo-planner/src/builder.rs:163-192).  COUNT -> count; SUM -> sum; AVG -> (count u64, sum f64).
void WindowAggOp::export_partial(OutSet* os, int64_t n, BatchesPriv* out) {
  std::vector<OutColumn> cols;
  std::vector<size_t> fix_f64;  // AVG state kept as an exact integer sum: the partial schema wants Float64
  if (keyed_) {
    OutColumn k;
    k.name = "key";
    k.format = key_format_;
    k.data = d2h_column(os->key.p, n, stream_, &st_.d2h_bytes);
    cols.push_back(k);
  }
  for (int g = 0; g < n_aggs_; ++g) {
    auto add = [&](const char* nm, const char* fmt, const void* dev) {
      OutColumn c;
      c.name = std::string("agg") + std::to_string(g) + nm;
      c.format = fmt;
      c.data = d2h_column(dev, n, stream_, &st_.d2h_bytes);
      cols.push_back(c);
    };
    switch (agg_kind_[g]) {
      case ARROYO_B200_AGG_COUNT_STAR: add("[count]", "l", os->state[0].p); break;
      case ARROYO_B200_AGG_SUM_I64: add("[sum]", "l", os->state[agg_acc_[g]].p); break;
      case ARROYO_B200_AGG_AVG_I64:
        add("[count]", "L", os->state[0].p);
        add("[sum]", "g", os->state[agg_acc_[g]].p);
        if (acc_kind_[agg_acc_[g]] == ACC_SUM_I64) fix_f64.push_back(cols.size() - 1);
        break;
      case ARROYO_B200_AGG_MIN_I64: add("[min]", agg_format_[g].c_str(), os->state[agg_acc_[g]].p); break;
      case ARROYO_B200_AGG_MAX_I64: add("[max]", agg_format_[g].c_str(), os->state[agg_acc_[g]].p); break;
    }
  }
  OutColumn t;
  t.name = "_timestamp";
  t.format = "tsn:";
  t.data = d2h_column(os->ts.p, n, stream_, &st_.d2h_bytes);
  cols.push_back(t);
  AB_CUDA(cudaStreamSynchronize(stream_));
  for (size_t ci : fix_f64) {
    long long* raw = (long long*)cols[ci].data;
    double* d = (double*)cols[ci].data;
    for (int64_t i = 0; i < n; ++i) d[i] = (double)raw[i];
  }
  out->arrays.emplace_back();
  out->schemas.emplace_back();
  export_batch(cols, n, &out->arrays.back(), &out->schemas.back());
}

void WindowAggOp::emit_window(int64_t a, int64_t b, size_t out_index, BatchesPriv* out_host,
                              std::vector<ArroyoB200DeviceBatch>* out_dev) {
  // panes of the window = window store (tier) restricted to [a, b)   (sliding :161-168)
  std::vector<int64_t> members;
  for (auto it = panes_.lower_bound(a); it != panes_.end() && it->first < b; ++it)
    if (it->second.in_tier) members.push_back(it->first);
  if (avg_exact_ && guard_vals_) {
    uint64_t window_rows = 0;
    for (int64_t m : members) window_rows += panes_.at(m).rows;
    if (window_rows >= (1ull << 32)) promote_avg();
  }
  std::vector<const unsigned long long*> blocks;
  int n_add = 0;
  bool use_running = false;
  if (running_mode_) {
    if (!running_) {
      running_ = acquire_block();
      // W starts from all-zero (identity of the invertible accumulators)
    }
    std::set<int64_t> target(members.begin(), members.end());
    std::vector<const unsigned long long*> add, sub;
    for (int64_t m : target)
      if (!in_running_.count(m)) {
        const Pane& p = panes_.at(m);
        add.push_back(p.dev);
        if (p.frozen) add.push_back(p.frozen);
      }
    for (int64_t m : in_running_)
      if (!target.count(m)) {
        auto zi = zombies_.find(m);
        const Pane& p = zi != zombies_.end() ? zi->second : panes_.at(m);
        sub.push_back(p.dev);
        if (p.frozen) sub.push_back(p.frozen);
      }
    blocks = add;
    n_add = (int)add.size();
    blocks.insert(blocks.end(), sub.begin(), sub.end());
    in_running_ = target;
    use_running = true;
    if (target.empty()) {
      // nothing in the window: W is all zero by construction; nothing to emit
      if (blocks.empty()) return;
    }
  } else {
    for (int64_t m : members) {
      const Pane& p = panes_.at(m);
      blocks.push_back(p.dev);
      if (p.frozen) blocks.push_back(p.frozen);
    }
    if (blocks.empty()) return;  // aggregate over an empty input has no groups
  }
  // device output and asynchronous host output keep every window of the emission alive until the caller (or the
  // copy stream) is done with it: one output set per window; blocking host output reuses set 0
  OutSet* os = out_set(out_dev || async_out_ ? out_index : 0, std::max<uint64_t>(n_keys_host_, 1));
  const int64_t ts = cfg.final_projection ? b - 1 : a;
  int64_t n = run_emit(blocks, n_add, use_running, false, a, b, ts, os);
  // blocks of panes that had already left the store have now been subtracted from W
  for (auto& z : zombies_) {
    release_block(z.second.dev);
    release_block(z.second.frozen);
  }
  zombies_.clear();
  if (n == 0) return;
  if (n > 0) {  // (a deferred count is accounted for when it is resolved)
    st_.rows_out += (uint64_t)n;
    ++st_.windows_out;
  }
  if (out_host) {
    export_window(os, n, out_host);
  } else {
    ArroyoB200DeviceBatch d{};
    d.n_rows = n;
    int c = 0;
    std::vector<uint64_t> cols;
    if (keyed_) cols.push_back((uint64_t)os->key.p);
    for (int g = 0; g < n_aggs_; ++g) cols.push_back((uint64_t)os->agg[g].p);
    if (cfg.final_projection) {
      int wi = std::min<int>(std::max<int>(cfg.window_index, 0), (int)cols.size());
      cols.insert(cols.begin() + wi, (uint64_t)os->wend.p);
      cols.insert(cols.begin() + wi, (uint64_t)os->wstart.p);
    }
    cols.push_back((uint64_t)os->ts.p);
    for (uint64_t v : cols) d.cols[c++] = v;
    d.n_cols = c;
    out_dev->push_back(d);
  }
}

void WindowAggOp::handle_watermark(int64_t wm, BatchesPriv* out_host, std::vector<ArroyoB200DeviceBatch>* out_dev) {
  set_device();
  if (!defer_counts_) resolve_deferred();
  wait_outputs();
  launch_pending();
  sync_all();
  poll_releases(false);
  std::vector<PlanStep> steps;
  if (sliding_) sliding_planner_->watermark(wm, steps);
  else tumbling_->watermark(wm, steps);
  size_t out_index = 0;
  for (const PlanStep& s : steps) {
    switch (s.kind) {
      case PlanStep::JOIN: {
        auto it = panes_.find(s.a);
        AB_REQUIRE(it != panes_.end(), ARROYO_B200_RUNTIME, "closing a pane that is not resident");
        it->second.in_tier = true;
        break;
      }
      case PlanStep::EMIT: {
        if (!sliding_) {
          // tumbling: the popped bin is the whole window (tumbling :340-385)
          auto it = panes_.find(s.c);
          AB_REQUIRE(it != panes_.end(), ARROYO_B200_RUNTIME, "emitting a pane that is not resident");
          it->second.in_tier = true;
          emit_window(s.a, s.b, out_index++, out_host, out_dev);
          drop_pane(s.c);
        } else {
          emit_window(s.a, s.b, out_index++, out_host, out_dev);
        }
        break;
      }
      case PlanStep::LEAVE: {
        if (running_mode_ && in_running_.count(s.a)) {
          // W still contains this pane: keep its blocks until the next emit subtracts them in the
          // same pass that adds the entering pane (one kernel per slide)
          auto it = panes_.find(s.a);
          Pane z = it->second;
          it->second.dev = nullptr;
          it->second.frozen = nullptr;
          z.slot = -1;
          zombies_[s.a] = z;
        }
        drop_pane(s.a);
        break;
      }
      default:
        break;
    }
  }
  // bins below bin(watermark) are late from now on (tumbling :282-291, sliding :631-633)
  int64_t new_late = bin_start(wm, slide_);
  if (new_late > late_bin_) late_bin_ = new_late;
  // panes that were made resident ahead of time but can no longer receive rows
  std::vector<int64_t> dead;
  const auto& execs = sliding_ ? sliding_planner_->execs() : tumbling_->execs();
  for (auto& kv : panes_)
    if (kv.first < late_bin_ && !kv.second.in_tier && !execs.count(kv.first)) dead.push_back(kv.first);
  for (int64_t b : dead) drop_pane(b);
  // Panes below the late bin can no longer receive rows: they give their ring slot back (the block stays with the
  // pane).  The ring then only ever spans [late bin, newest bin], so a pane the planner never visits again -- the
  // reference leaks those too (sliding :176-187) -- cannot collide with a pane 4096 slides later.
  for (auto& kv : panes_) {
    if (kv.first >= late_bin_) break;
    Pane& p = kv.second;
    if (p.slot < 0) continue;
    h_pane_bins_[p.slot] = FREE_BIN;
    h_pane_ptrs_[p.slot] = nullptr;
    p.slot = -1;
    ring_dirty_ = true;
  }
  // make the pane at the watermark resident so the next rows do not defer
  if (wm != INT64_MAX && max_bin_seen_ != LLONG_MIN) {
    if (!panes_.count(late_bin_)) {
      uint32_t slot = (uint32_t)((uint64_t)late_bin_ / (uint64_t)slide_) & (ring_ - 1);
      if (h_pane_bins_[slot] == FREE_BIN && late_bin_ <= max_bin_seen_ + 2 * slide_) ensure_pane(late_bin_);
    }
  }
  if (!defer_counts_) collect_emit_times();
}

// handle_watermark for device-resident output without its last host wait: the emit kernels, the counter resets and the
// copies of the windows' row counts are enqueued and the call returns; poll_watermark_device (or any later entry
// point that needs the operator's state settled) reads the counts.  What the caller does in between -- typically
// handing over and submitting the next batches -- runs while the emission executes.
void WindowAggOp::begin_watermark_device(int64_t wm) {
  set_device();
  resolve_deferred();
  AB_REQUIRE(pending_dev.empty(), ARROYO_B200_INVALID_ARGUMENT,
             "the previous emission has not been collected (handle_watermark_device_poll)");
  if (!counts_done_) AB_CUDA(cudaEventCreateWithFlags(&counts_done_, cudaEventDisableTiming));
  struct Flag {
    bool& f;
    explicit Flag(bool& x) : f(x) { f = true; }
    ~Flag() { f = false; }
  } flag(defer_counts_);
  count_slots_used_ = 0;
  try {
    handle_watermark(wm, nullptr, &pending_dev);
  } catch (...) {
    if (counts_pending_) cudaEventRecord(counts_done_, stream_);
    throw;
  }
  if (counts_pending_) AB_CUDA(cudaEventRecord(counts_done_, stream_));
}

// Reads the row counts of a deferred emission (idempotent); empty windows are dropped like the blocking path drops them.
void WindowAggOp::resolve_deferred() {
  if (!counts_pending_) return;
  AB_CUDA(cudaEventSynchronize(counts_done_));
  counts_pending_ = false;
  const unsigned int* h = h_out_counts_.as<unsigned int>();
  std::vector<ArroyoB200DeviceBatch> kept;
  for (ArroyoB200DeviceBatch& d : pending_dev) {
    if (d.n_rows < 0) {
      const int slot = (int)(-d.n_rows - 1);
      d.n_rows = (int64_t)h[slot];
      if (d.n_rows) {
        st_.rows_out += (uint64_t)d.n_rows;
        ++st_.windows_out;
      }
    }
    if (d.n_rows) kept.push_back(d);
  }
  pending_dev.swap(kept);
  if (count_slots_used_ > 0) out_count_base_ = h[count_slots_used_ - 1];  // the counter's value after its last restart
  count_slots_used_ = 0;
  collect_emit_times();
}

void WindowAggOp::poll_watermark_device(std::vector<ArroyoB200DeviceBatch>* out) {
  set_device();
  resolve_deferred();
  out->swap(pending_dev);
  pending_dev.clear();
}

// Adds up the emit kernels' CUDA-event times (FLAG_PROFILE); the events go back to the pool.
void WindowAggOp::collect_emit_times() {
  if (!profile_ || emit_events_used_ == 0) return;
  AB_CUDA(cudaEventSynchronize(emit_events_[emit_events_used_ - 1].second));
  for (size_t i = 0; i < emit_events_used_; ++i) {
    float ms = 0;
    AB_CUDA(cudaEventElapsedTime(&ms, emit_events_[i].first, emit_events_[i].second));
    st_.emit_ms += ms;
  }
  emit_events_used_ = 0;
}

void WindowAggOp::handle_checkpoint(int64_t wm, BatchesPriv* out) {
  set_device();
  resolve_deferred();
  wait_outputs();
  launch_pending();
  sync_all();
  std::vector<PlanStep> steps;
  if (sliding_) sliding_planner_->checkpoint(wm != INT64_MIN, wm, steps);
  else tumbling_->checkpoint(steps);
  for (const PlanStep& s : steps) {
    if (s.kind != PlanStep::CHECKPOINT_PANE) continue;
    auto it = panes_.find(s.a);
    AB_REQUIRE(it != panes_.end(), ARROYO_B200_RUNTIME, "checkpointing a pane that is not resident");
    Pane& p = it->second;
    OutSet* os = out_set(0, std::max<uint64_t>(n_keys_host_, 1));
    // the rows received since the last drain = the active block (the reference drains the running
    // Partial exec and writes its output, sliding :705-733)
    int64_t n = run_emit({p.dev}, 1, false, true, 0, 0, s.a, os);
    if (n > 0) export_partial(os, n, out);
    // fold into the frozen block so the next checkpoint writes only new rows
    p.delta_exported = true;
    if (!p.frozen) p.frozen = acquire_block();
    FoldParams fp{};
    fp.active = p.dev;
    fp.frozen = p.frozen;
    fp.id_cap = id_cap_;
    fp.n_ids = n_keys_host_;
    fp.n_acc = n_acc_;
    for (int a = 0; a < n_acc_; ++a) fp.acc_kind[a] = acc_kind_[a];
    int grid = (int)std::min<uint32_t>((n_keys_host_ + 255) / 256, (uint32_t)num_sms_ * 8);
    fold_kernel<<<std::max(grid, 1), 256, 0, stream_>>>(fp);
    AB_CUDA(cudaGetLastError());
    ++st_.kernel_launches;
  }
  // Panes that closed since the last checkpoint: the reference inserts their partial batches into table
  // "t" when it closes them (sliding :133-158); here they stay on the device and are handed to the shim
  // at the checkpoint, which is when the table is persisted -- restore sees the same table contents.
  for (auto& kv : panes_) {
    Pane& p = kv.second;
    if (!p.in_tier || p.exported) continue;
    // what the table does not have yet: the active block, plus the frozen one unless an earlier
    // checkpoint (or the restore) already wrote it
    std::vector<const unsigned long long*> blocks{p.dev};
    if (p.frozen && !p.delta_exported) blocks.push_back(p.frozen);
    OutSet* os = out_set(0, std::max<uint64_t>(n_keys_host_, 1));
    int64_t n = run_emit(blocks, (int)blocks.size(), false, true, 0, 0, kv.first, os);
    if (n > 0) export_partial(os, n, out);
    p.exported = true;
  }
  AB_CUDA(cudaStreamSynchronize(stream_));
  collect_emit_times();
}

// Restore (tumbling :228-248, sliding :556-595): partial batches go back into pane blocks.
void WindowAggOp::on_start(ArrowArray* state, ArrowSchema* schemas, int64_t n, int64_t watermark, int64_t table_min) {
  set_device();
  const bool has_wm = watermark != INT64_MIN;
  if (has_wm) late_bin_ = std::max<int64_t>(late_bin_, bin_start(watermark, slide_));
  if (sliding_) sliding_planner_->restore_begin(has_wm, watermark);
  // expected partial layout
  int n_state_cols = 0;
  for (int g = 0; g < n_aggs_; ++g) n_state_cols += agg_kind_[g] == ARROYO_B200_AGG_AVG_I64 ? 2 : 1;
  const int expect_cols = (keyed_ ? 1 : 0) + n_state_cols + 1;
  std::vector<DevBuf> keep;
  for (int64_t bi = 0; bi < n; ++bi) {
    int64_t rows = 0;
    std::vector<InColumn> cols = import_batch(&state[bi], &schemas[bi], &rows);
    AB_REQUIRE((int)cols.size() == expect_cols, ARROYO_B200_INVALID_ARGUMENT,
               "state batch does not match the partial schema");
    if (rows == 0) continue;
    if (keyed_) key_format_ = cols[0].format;
    const int64_t ts = (int64_t)cols.back().data[0];
    const int64_t bin = bin_start(ts, slide_);
    ensure_pane(bin);
    Pane& p = panes_.at(bin);
    if (!p.frozen) p.frozen = acquire_block();
    bool to_tier = false;
    if (sliding_) to_tier = sliding_planner_->restore_pane(ts);
    else tumbling_->restore(bin);
    if (to_tier) p.in_tier = true;
    p.exported = to_tier;
    p.delta_exported = true;
    // upload columns
    PartialParams pp{};
    pp.n = rows;
    pp.keyed = keyed_ ? 1 : 0;
    pp.n_acc = n_acc_;
    for (int a = 0; a < n_acc_; ++a) pp.acc_kind[a] = acc_kind_[a];
    auto up = [&](const uint64_t* h) -> const unsigned long long* {
      keep.emplace_back((size_t)rows * 8);
      AB_CUDA(cudaMemcpyAsync(keep.back().p, h, (size_t)rows * 8, cudaMemcpyHostToDevice, stream_));
      return keep.back().as<unsigned long long>();
    };
    int ci = 0;
    if (keyed_) pp.key = (const long long*)up(cols[ci++].data);
    for (int a = 0; a < MAX_ACC; ++a) pp.state[a] = nullptr;
    std::vector<std::pair<int, int>> avg_sum_cols;  // (agg, column of its f64 sum)
    for (int g = 0; g < n_aggs_; ++g) {
      switch (agg_kind_[g]) {
        case ARROYO_B200_AGG_COUNT_STAR: {
          const unsigned long long* c = up(cols[ci++].data);
          if (!pp.state[0]) pp.state[0] = c;
          break;
        }
        case ARROYO_B200_AGG_AVG_I64: {
          const unsigned long long* c = up(cols[ci++].data);
          if (!pp.state[0]) pp.state[0] = c;
          avg_sum_cols.emplace_back(g, ci++);
          break;
        }
        default:
          pp.state[agg_acc_[g]] = up(cols[ci++].data);
          break;
      }
    }
    std::vector<long long> conv;
    for (auto& pr : avg_sum_cols) {
      const int acc = agg_acc_[pr.first];
      if (acc_kind_[acc] == ACC_SUM_F64) {
        pp.state[acc] = up(cols[pr.second].data);
      } else if (!pp.state[acc]) {
        // exact-sum AVG without a SUM over the same column: the checkpoint only has the f64 image of the sum
        // (exact below 2^53); a SUM column, when present, already restored the integer accumulator above
        conv.resize((size_t)rows);
        const double* d = (const double*)cols[pr.second].data;
        for (int64_t i = 0; i < rows; ++i) conv[(size_t)i] = (long long)__builtin_llround(d[i]);
        keep.emplace_back((size_t)rows * 8);
        AB_CUDA(cudaMemcpyAsync(keep.back().p, conv.data(), (size_t)rows * 8, cudaMemcpyHostToDevice, stream_));
        AB_CUDA(cudaStreamSynchronize(stream_));
        pp.state[acc] = keep.back().as<unsigned long long>();
      }
    }
    if (pp.state[0] == nullptr) {
      // SUM / MIN / MAX-only plans carry no row count in their partial state; the rows accumulator is only the
      // "this key is present in the pane" flag for them, so every restored state row counts as one
      std::vector<unsigned long long> ones((size_t)rows, 1ull);
      keep.emplace_back((size_t)rows * 8);
      AB_CUDA(cudaMemcpyAsync(keep.back().p, ones.data(), (size_t)rows * 8, cudaMemcpyHostToDevice, stream_));
      AB_CUDA(cudaStreamSynchronize(stream_));
      pp.state[0] = keep.back().as<unsigned long long>();
    }
    // room for every key of the batch at the target bucket fill (most of them are usually known already)
    while (keyed_ && (uint64_t)total_keys_host_ + (uint64_t)rows > n_buckets_ * (uint64_t)BD_MEAN) {
      AB_CUDA(cudaStreamSynchronize(stream_));
      grow_ids();
    }
    pp.dict = dict_view();
    pp.pane = panes_.at(bin).frozen;
    pp.id_cap = id_cap_;
    pp.counters = d_counters();
    int grid = (int)std::min<int64_t>((rows + 255) / 256, (int64_t)num_sms_ * 8);
    ingest_partial_kernel<<<std::max(grid, 1), 256, 0, stream_>>>(pp);
    AB_CUDA(cudaGetLastError());
    ++st_.kernel_launches;
    Counters c{};
    AB_CUDA(cudaMemcpyAsync(&c, book_.p, sizeof c, cudaMemcpyDeviceToHost, stream_));
    AB_CUDA(cudaStreamSynchronize(stream_));
    AB_REQUIRE(c.lost == 0, ARROYO_B200_RUNTIME, "dictionary overflow during restore");
    total_keys_host_ = c.n_keys;
    last_counters_ = c;
    max_bin_seen_ = std::max<int64_t>(max_bin_seen_, bin);
    if (state[bi].release) state[bi].release(&state[bi]);
  }
  if (sliding_) sliding_planner_->restore_end(table_min != INT64_MIN, table_min);
  AB_CUDA(cudaStreamSynchronize(stream_));
}

void WindowAggOp::stats(ArroyoB200Stats* out) {
  set_device();
  resolve_deferred();  // an outstanding emission's windows are counted once their row counts are in
  st_.n_keys = keyed_ ? total_keys_host_ : 0;
  st_.rows_late = last_counters_.late_rows;
  *out = st_;
}

}  // namespace

OpBase* make_window_agg_op(const ArroyoB200OpConfig& cfg) { return new WindowAggOp(cfg); }

}  // namespace ab
