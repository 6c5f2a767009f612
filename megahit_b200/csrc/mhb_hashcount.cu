// mhb_hashcount.cu -- solid-edge counting by radix PARTITION + per-bucket HASH AGGREGATION (A4 + A5 for 8-byte count
// records, i.e. k <= 28), an alternative to "sort all records by all 7 key bytes, then run-length count".
//
// Why: the run-length count (kmer_counter.cpp:254-305) needs equal (k+1)-mers to meet, not a total order of the 1.23 G
// records; only the SOLID edges (5 % of the distinct ones on the bench workload) have to come out sorted.  So:
//   1. three stable radix passes on the three leading key bytes (the same k_radix_pass3 the sort uses) group the
//      records by their leading 24 key bits - 3 x 2NS bytes instead of 7 x 2NS;
//   2. k_bucket_bounds finds the 65 537 boundaries of the reference's 16-bit buckets (base_engine.h kNumBuckets) by
//      binary search, and k_slice_table cuts every bucket into slices of ~6000 records whose boundaries are moved to
//      the next change of the 24-bit prefix: a slice is contiguous and key-closed;
//   3. k_hash_count: a CTA takes a slice and aggregates it in a shared-memory open-addressing table keyed by the
//      remaining 42 record bits: occurrence counts first, then, for the keys that reached the solid threshold, the
//      4 + 4 prev/next tallies (has_in / has_out, :279-305) in a second sweep over the same records (L2 hits); the solid
//      keys of the slice (a few hundred) are ordered by a counting sort in shared memory and appended to the slice's
//      area of a scratch list.  A slice with more distinct keys than the table holds is split into four key
//      sub-ranges, recursively (the slice is re-streamed per sub-range) - correctness never depends on the key
//      distribution, only speed does;
//   4. a scan over the per-slice solid counts + k_hash_gather write the `.edges`-format records (PackEdge, :32-52),
//      the aux flags and the multiplicity histogram exactly as mhb_count_solid does.
// Output is bit-identical to sort + mhb_count_solid (tests/test_gpu_parity.py).  HBM traffic of the count stage falls
// from (7 x 2 + 1) NS to (3 x 2 + 1) NS bytes.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include "mhb.h"
#include "mhb_common.cuh"
#include "mhb_count.cuh"

using namespace mhb;

namespace {

constexpr int kHcHist = 1024;                  // multiplicities < kHcHist are histogrammed in shared memory
constexpr u64 kHcEmpty = ~0ull;
constexpr int kHcBatch = 4;                    // records per thread in flight while streaming a slice
constexpr u32 kRemBits = 42;                   // record bits 47..6
constexpr u32 kHcHotCount = 256;               // keys this frequent may wrap a byte tally: they get exact 32-bit tallies
constexpr int kHcHotRound = 32;                // ... this many at a time
constexpr int kHcMaxProbes = 48;               // longer probe sequences = the table is too full for this sub-range
constexpr int kHcStack = 72;

__device__ __forceinline__ u64 rec_key64(const uint2 r) { return ((u64)r.x << 32) | r.y; }

// bounds[b] = first record whose 16-bit prefix is >= b (b = 0..65536); the records are sorted on that prefix
__global__ void k_bucket_bounds(const uint2 *__restrict__ recs, u64 n, u64 *__restrict__ bounds) {
  const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b > 65536u) return;
  u64 lo = 0, hi = n;
  while (lo < hi) {
    const u64 mid = (lo + hi) >> 1;
    if ((recs[mid].x >> 16) < b) lo = mid + 1;
    else hi = mid;
  }
  bounds[b] = lo;
}

// Geometry of the hash kernel: THREADS per CTA, 2^LOG_SLOTS table slots, CTAS per SM.  The per-slice fixed costs
// (barriers, table sweeps, the ordering scan) are amortised over more records by the larger geometries.
template <int THREADS_, int LOG_SLOTS_, int CTAS_>
struct HcGeom {
  static constexpr int THREADS = THREADS_, LOG_SLOTS = LOG_SLOTS_, SLOTS = 1 << LOG_SLOTS_, CTAS = CTAS_;
  static constexpr int MAX_SOLID = SLOTS / 4;   // solid keys per sub-range (ordering buffers)
  static constexpr int CELLS = 2 * THREADS;     // counting-sort cells that order a sub-range's solid keys
  static constexpr int LOG_CELLS = LOG_SLOTS_ - 2 >= 0 ? (THREADS_ == 256 ? 9 : (THREADS_ == 512 ? 10 : 11)) : 9;
  static constexpr u32 SLICE = (u32)(SLOTS * 1.83);  // records per slice: ~0.68 x SLOTS distinct keys on 30x reads (swept)
};

template <class G>
struct HcShared {
  u64 keys[G::SLOTS];
  u32 cnt[G::SLOTS];           // occurrences
  u32 pt[G::SLOTS];            // prev tallies, one byte per base (exact while the key has < 256 occurrences)
  u32 nt[G::SLOTS];            // next tallies
  u64 sorted[G::MAX_SOLID];    // rem42 << 22 | cnt16 << 6 | aux
  u64 tmp[G::MAX_SOLID];
  u32 cell_base[G::CELLS];
  u32 cell_cur[G::CELLS];
  u32 cta_hist[kHcHist];
  u32 wide[kHcHotRound][8];    // exact tallies of the hot keys of the current round
  uint16_t hot_slot[G::MAX_SOLID];
  u64 st_prefix[kHcStack];
  u32 st_bits[kHcStack];
  u32 warp_sum[G::THREADS / 32];
  u32 n_solid, n_hot, overflow, bucket, out_cursor, sp;
};

__device__ __forceinline__ u32 lane_lt_mask() { return (1u << (threadIdx.x & 31)) - 1u; }

// plain shared-memory reduction.  nvcc turns atomicAdd() on shared memory whose result is unused into a
// MATCH.ANY-driven loop over the groups of lanes that hit the same address; with ~1 lane per address that is overhead.
__device__ __forceinline__ void smem_add(u32 *p, u32 v) {
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"((u32)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}

template <class G>
__device__ __forceinline__ u32 hc_hash(u64 r) { return (u32)((r * 0x9E3779B97F4A7C15ull) >> (64 - G::LOG_SLOTS)); }

// slot of key r, inserting it when absent.  Returns SLOTS when the probe sequence gets too long: the sub-range holds
// too many distinct keys for the table (the caller flags overflow and the sub-range is split).
template <class G>
__device__ __forceinline__ u32 hc_insert(HcShared<G> &s, u64 r) {
  u32 h = hc_hash<G>(r);
  for (int probes = 0; probes < kHcMaxProbes; ++probes) {
    u64 cur = s.keys[h];
    if (cur == r) return h;
    if (cur == kHcEmpty) {
      cur = atomicCAS((unsigned long long *)&s.keys[h], kHcEmpty, r);
      if (cur == kHcEmpty || cur == r) return h;
    }
    h = (h + 1) & (G::SLOTS - 1);
  }
  return G::SLOTS;
}
template <class G>
__device__ __forceinline__ u32 hc_find(const HcShared<G> &s, u64 r) {
  u32 h = hc_hash<G>(r);
  while (s.keys[h] != r) h = (h + 1) & (G::SLOTS - 1);
  return h;
}

// take the multiplicity histogram contribution of the occupied slots back (a sub-range that has to be split after
// it was judged)
template <class G>
__device__ __forceinline__ void hc_hist_undo(HcShared<G> &s, u64 *mul_hist) {
  for (u32 i = threadIdx.x; i < (u32)G::SLOTS; i += G::THREADS) {
    if (s.keys[i] == kHcEmpty) continue;
    const u32 c = s.cnt[i];
    const u32 c16 = c > 65535u ? 65535u : c;
    if (c16 < (u32)kHcHist) atomicAdd(&s.cta_hist[c16], 0xFFFFFFFFu);
    else atomicAdd((unsigned long long *)&mul_hist[c16], ~0ull);
  }
}

// exclusive scan of s.cell_base[0 .. CELLS) in place (CELLS = 2 * THREADS); also primes cell_cur
template <class G>
__device__ __forceinline__ void hc_scan_cells(HcShared<G> &s) {
  const u32 t = threadIdx.x, lane = t & 31, w = t >> 5;
  const u32 a = s.cell_base[2 * t], b = s.cell_base[2 * t + 1];
  u32 v = a + b;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const u32 o = __shfl_up_sync(0xffffffffu, v, d);
    if ((int)lane >= d) v += o;
  }
  if (lane == 31) s.warp_sum[w] = v;
  __syncthreads();
  if (w == 0) {
    u32 x = lane < G::THREADS / 32 ? s.warp_sum[lane] : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 o = __shfl_up_sync(0xffffffffu, x, d);
      if ((int)lane >= d) x += o;
    }
    if (lane < G::THREADS / 32) s.warp_sum[lane] = x;  // inclusive
  }
  __syncthreads();
  const u32 excl = v - (a + b) + (w ? s.warp_sum[w - 1] : 0u);
  s.cell_base[2 * t] = excl;
  s.cell_base[2 * t + 1] = excl + a;
  s.cell_cur[2 * t] = excl;
  s.cell_cur[2 * t + 1] = excl + a;
  __syncthreads();
}

__device__ __forceinline__ bool hc_any_byte_ge(u32 w, u32 m) {
  return (w & 0xFFu) >= m || ((w >> 8) & 0xFFu) >= m || ((w >> 16) & 0xFFu) >= m || (w >> 24) >= m;
}

// Slice table: bucket b (16-bit prefix) is cut into ceil(n_b / T) slices whose boundaries are moved forward to the next
// change of the 24-bit prefix, so that a slice is a contiguous, key-closed range (records with equal keys share their
// prefix, so they never straddle such a boundary).  slice_off[b] = first slice id of bucket b (exclusive scan of the
// per-bucket slice counts).  One thread per slice: slice_start[s] = first record of slice s, slice_start[n_slices] = n
// (the end of a slice is the start of the next one), slice_bucket[s] = its bucket, slice_base[s] = where its solid
// entries go in the scratch list: list[a_s / m + s ...) with a_s the slice's first record (a slice of n records holds at
// most n / m solid keys and floor is super-additive: the areas never overlap).  Computed up front so that a hash CTA
// starts a slice with two loads instead of a serial search and block-wide boundary scans.
__global__ void k_slice_table(const uint2 *__restrict__ recs, const u64 *__restrict__ bounds, const u64 *__restrict__ slice_off,
                              const u64 *__restrict__ n_slices_dev, u64 n, int m, u64 *__restrict__ slice_start,
                              u64 *__restrict__ slice_base, u32 *__restrict__ slice_bucket) {
  const u64 sl = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  const u64 n_slices = *n_slices_dev;
  if (sl > n_slices) return;
  if (sl == n_slices) {
    slice_start[sl] = n;
    return;
  }
  u32 a = 0, z = 65536;  // bucket of this slice: last b with slice_off[b] <= sl
  while (z - a > 1) {
    const u32 mid = (a + z) >> 1;
    if (slice_off[mid] <= sl) a = mid;
    else z = mid;
  }
  const u32 b = a;
  const u64 blo = bounds[b], bhi = bounds[b + 1];
  const u64 n_in_b = slice_off[b + 1] - slice_off[b], idx = sl - slice_off[b];
  const u64 step = (bhi - blo + n_in_b - 1) / n_in_b;
  const u64 p = blo + idx * step;
  u64 lo;
  if (p <= blo) {
    lo = blo;
  } else if (p >= bhi) {
    lo = bhi;
  } else {  // first q in [p, bhi) whose 24-bit prefix exceeds that of record p - 1 (sorted on it), else bhi
    const u32 g = recs[p - 1].x >> 8;
    u64 l = p, h = bhi;
    while (l < h) {
      const u64 mid = (l + h) >> 1;
      if ((recs[mid].x >> 8) <= g) l = mid + 1;
      else h = mid;
    }
    lo = l;
  }
  slice_start[sl] = lo;
  slice_base[sl] = lo / (u64)m + sl;
  slice_bucket[sl] = b;
}

// Work unit = a slice of the slice table, taken by ticket (the next ticket is requested a whole slice ahead), read
// once with every lane busy.
// One sweep per slice: occurrence count and the 4 + 4 prev / next tallies (kmer_counter.cpp:279-295) of every key, the
// tallies as byte fields; only keys with >= 256 occurrences ("hot": a byte could wrap) get a second sweep with exact
// 32-bit tallies, 32 keys at a time.
template <class G>
__global__ void __launch_bounds__(G::THREADS, G::CTAS)
    k_hash_count(const uint2 *__restrict__ recs, const u64 *__restrict__ slice_start, const u64 *__restrict__ n_slices_dev,
                 int m, u32 *ticket, u64 *__restrict__ list, u32 *__restrict__ slice_count, u64 *mul_hist, u32 *err_flag) {
  constexpr int THREADS = G::THREADS, SLOTS = G::SLOTS, MAX_SOLID = G::MAX_SOLID, CELLS = G::CELLS;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  HcShared<G> &s = *reinterpret_cast<HcShared<G> *>(smem_raw);
  const u32 tid = threadIdx.x;
  for (u32 i = tid; i < kHcHist; i += THREADS) s.cta_hist[i] = 0;
  for (u32 i = tid; i < (u32)SLOTS; i += THREADS) {
    s.keys[i] = kHcEmpty;
    s.cnt[i] = 0;
    s.pt[i] = 0;
    s.nt[i] = 0;
  }
  __syncthreads();
  const u64 n_slices = *n_slices_dev;
  const u32 um = (u32)m;
  u32 next = tid == 0 ? atomicAdd(ticket, 1u) : 0u;
  while (true) {
    if (tid == 0) {
      s.bucket = next;
      next = atomicAdd(ticket, 1u);  // tickets only grow: once this one is past the end, so is the prefetched one
    }
    __syncthreads();
    const u32 sl = s.bucket;
    if (sl >= n_slices) break;
    const u64 lo = slice_start[sl], hi = slice_start[sl + 1];
    const u64 base = lo / (u64)m + sl;
    if (tid == 0) {
      s.out_cursor = 0;
      s.st_prefix[0] = 0;
      s.st_bits[0] = 0;
      s.sp = 1;
    }
    if (hi <= lo) {  // a 24-bit group longer than a slice swallowed this one
      if (tid == 0) slice_count[sl] = 0;
      __syncthreads();
      continue;
    }
    __syncthreads();
    while (s.sp > 0) {
      // ---------------- one key sub-range: the records whose remainder starts with `prefix` (`bits` bits) -------
      const u32 sp = s.sp - 1;
      const u64 prefix = s.st_prefix[sp];
      const u32 bits = s.st_bits[sp];
      __syncthreads();
      if (tid == 0) {
        s.sp = sp;
        s.n_solid = 0;
        s.n_hot = 0;
        s.overflow = 0;
      }
      __syncthreads();
      // ---- the sweep: occurrence counts and byte tallies ----
      for (u64 i0 = lo + tid; i0 < hi; i0 += (u64)THREADS * kHcBatch) {
        uint2 v[kHcBatch];
#pragma unroll
        for (int j = 0; j < kHcBatch; ++j) {
          const u64 i = i0 + (u64)j * THREADS;
          v[j] = i < hi ? recs[i] : make_uint2(0, 0);
        }
#pragma unroll
        for (int j = 0; j < kHcBatch; ++j) {
          const u64 i = i0 + (u64)j * THREADS;
          if (i >= hi) break;
          const u64 key = rec_key64(v[j]);
          const u64 r = (key >> 6) & ((1ull << kRemBits) - 1);
          if (bits && (r >> (kRemBits - bits)) != prefix) continue;
          const u32 h = hc_insert<G>(s, r);
          if (h == (u32)SLOTS) {
            s.overflow = 1;
            continue;
          }
          smem_add(&s.cnt[h], 1u);
          const u32 p = (u32)(key >> 3) & 7u, nx = (u32)key & 7u;
          if (p < 4) smem_add(&s.pt[h], 1u << (8 * p));
          if (nx < 4) smem_add(&s.nt[h], 1u << (8 * nx));
        }
        if (s.overflow) break;
      }
      __syncthreads();
      bool failed = s.overflow != 0;
      u32 ns = 0;
      if (!failed) {
        // ---- judge: multiplicity histogram; the keys that reached the solid threshold get a rank and their flags ----
        for (u32 i0 = 0; i0 < (u32)SLOTS; i0 += THREADS) {
          const u32 slot = i0 + tid;
          const bool on = s.keys[slot] != kHcEmpty;
          const u32 c = on ? s.cnt[slot] : 0u;
          const u32 c16 = c > 65535u ? 65535u : c;
          const u32 ones = __ballot_sync(0xffffffffu, on && c16 == 1u), twos = __ballot_sync(0xffffffffu, on && c16 == 2u);
          if (on && c16 > 2u) {
            if (c16 < (u32)kHcHist) smem_add(&s.cta_hist[c16], 1u);
            else atomicAdd((unsigned long long *)&mul_hist[c16], 1ull);
          }
          const bool solid = on && c >= um;
          const u32 sm_ = __ballot_sync(0xffffffffu, solid);
          u32 wbase = 0;
          if ((tid & 31) == 0) {
            if (ones) atomicAdd(&s.cta_hist[1], (u32)__popc(ones));
            if (twos) atomicAdd(&s.cta_hist[2], (u32)__popc(twos));
            if (sm_) wbase = atomicAdd(&s.n_solid, (u32)__popc(sm_));
          }
          wbase = __shfl_sync(0xffffffffu, wbase, 0);
          if (solid) {
            const u32 rank = wbase + __popc(sm_ & lane_lt_mask());
            if (rank < (u32)MAX_SOLID) {
              u64 e = (s.keys[slot] << 22) | ((u64)c16 << 6);
              if (c >= kHcHotCount) {  // byte tallies may have wrapped: exact tallies in a second sweep
                const u32 hi_ = atomicAdd(&s.n_hot, 1u);
                if (hi_ < (u32)MAX_SOLID) s.hot_slot[hi_] = (uint16_t)slot;
                s.pt[slot] = hi_;   // index among the hot keys
                s.nt[slot] = rank;  // where its entry lives
              } else {
                e |= (hc_any_byte_ge(s.pt[slot], um) ? 0ull : 1ull) | (hc_any_byte_ge(s.nt[slot], um) ? 0ull : 2ull);
              }
              s.sorted[rank] = e;
            }
          }
        }
        __syncthreads();
        ns = s.n_solid;
        if (ns > (u32)MAX_SOLID) {  // too many solid keys for the ordering buffers: take the histogram back, split
          hc_hist_undo<G>(s, mul_hist);
          failed = true;
        }
      }
      if (!failed && ns) {
        const u32 n_hot = s.n_hot;
        for (u32 h0 = 0; h0 < n_hot; h0 += kHcHotRound) {
          // ---- exact prev / next tallies of up to 32 hot keys: one more sweep over the slice ----
          for (u32 i = tid; i < (u32)kHcHotRound * 8; i += THREADS) s.wide[i >> 3][i & 7] = 0;
          __syncthreads();
          for (u64 i0 = lo + tid; i0 < hi; i0 += (u64)THREADS * kHcBatch) {
            uint2 v[kHcBatch];
#pragma unroll
            for (int j = 0; j < kHcBatch; ++j) {
              const u64 i = i0 + (u64)j * THREADS;
              v[j] = i < hi ? recs[i] : make_uint2(0, 0);
            }
#pragma unroll
            for (int j = 0; j < kHcBatch; ++j) {
              const u64 i = i0 + (u64)j * THREADS;
              if (i >= hi) break;
              const u64 key = rec_key64(v[j]);
              const u64 r = (key >> 6) & ((1ull << kRemBits) - 1);
              if (bits && (r >> (kRemBits - bits)) != prefix) continue;
              const u32 slot = hc_find<G>(s, r);
              const u32 c = s.cnt[slot];
              if (c < kHcHotCount || c < um) continue;
              const u32 hidx = s.pt[slot] - h0;
              if (hidx >= (u32)kHcHotRound) continue;
              const u32 p = (u32)(key >> 3) & 7u, nx = (u32)key & 7u;
              if (p < 4) smem_add(&s.wide[hidx][p], 1u);
              if (nx < 4) smem_add(&s.wide[hidx][4 + nx], 1u);
            }
          }
          __syncthreads();
          for (u32 i = tid; i < (u32)kHcHotRound && h0 + i < n_hot; i += THREADS) {
            bool has_in = false, has_out = false;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              has_in = has_in || s.wide[i][c] >= um;
              has_out = has_out || s.wide[i][4 + c] >= um;
            }
            s.sorted[s.nt[s.hot_slot[h0 + i]]] |= (has_in ? 0ull : 1ull) | (has_out ? 0ull : 2ull);
          }
          __syncthreads();
        }
        // ---- order the solid keys: counting sort on the next key bits, ties ranked inside their cell ----
        for (u32 i = tid; i < (u32)CELLS; i += THREADS) s.cell_base[i] = 0;
        __syncthreads();
        const u32 cshift = 22 + (kRemBits - G::LOG_CELLS);  // entry bits 63..22 hold the remainder
        for (u32 i = tid; i < ns; i += THREADS) smem_add(&s.cell_base[(u32)((s.sorted[i] << bits) >> cshift)], 1u);
        __syncthreads();
        hc_scan_cells<G>(s);
        for (u32 i = tid; i < ns; i += THREADS) {
          const u64 e = s.sorted[i];
          s.tmp[atomicAdd(&s.cell_cur[(u32)((e << bits) >> cshift)], 1u)] = e;
        }
        __syncthreads();
        const u32 at = s.out_cursor;
        for (u32 i = tid; i < ns; i += THREADS) {
          const u64 e = s.tmp[i];
          const u32 c = (u32)((e << bits) >> cshift);
          const u32 b0 = s.cell_base[c], b1 = c + 1 < (u32)CELLS ? s.cell_base[c + 1] : ns;
          u32 r = b0;
          for (u32 j = b0; j < b1; ++j) r += s.tmp[j] < e ? 1u : 0u;
          list[base + at + r] = e;
        }
        __syncthreads();
        if (tid == 0) s.out_cursor = at + ns;
      }
      // ---- clear the table ----
      for (u32 i = tid; i < (u32)SLOTS; i += THREADS) {
        s.keys[i] = kHcEmpty;
        s.cnt[i] = 0;
        s.pt[i] = 0;
        s.nt[i] = 0;
      }
      __syncthreads();
      if (tid == 0 && failed) {  // split this sub-range in four (ascending order is kept: the smallest child is popped first)
        if (bits + 2 > kRemBits || s.sp + 4 > (u32)kHcStack) atomicExch(err_flag, 1u);
        else
          for (int c = 3; c >= 0; --c) {
            s.st_prefix[s.sp] = (prefix << 2) | (u64)c;
            s.st_bits[s.sp] = bits + 2;
            ++s.sp;
          }
      }
      __syncthreads();
    }
    // ---- the slice is complete ----
    if (tid == 0) slice_count[sl] = s.out_cursor;
    __syncthreads();
  }
  for (u32 i = tid; i < kHcHist; i += THREADS)
    if (s.cta_hist[i]) atomicAdd((unsigned long long *)&mul_hist[i], (unsigned long long)s.cta_hist[i]);
}

// 512 threads, 4096 slots, 2 CTAs/SM: geometry B of the sweep in profiles/r2e_* (256 x 2048 x 3 and 1024 x 8192 x 1, at
// their own and at other slice sizes, were slower)
using HcGeomB = HcGeom<512, 12, 2>;

// per-bucket slice counts: ceil(n_b / T) (0 for an empty bucket)
__global__ void k_slice_counts(const u64 *__restrict__ bounds, u32 T, u32 *__restrict__ cnt) {
  const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= 65536u) return;
  const u64 nb = bounds[b + 1] - bounds[b];
  cnt[b] = (u32)((nb + T - 1) / T);
}

// PackEdge (kmer_counter.cpp:32-52): every slice's ordered solid entries -> `.edges` records + aux flags, in slice
// (= key) order
__global__ void __launch_bounds__(256)
    k_hash_gather(const u64 *__restrict__ list, const u64 *__restrict__ n_slices_dev, const u32 *__restrict__ slice_count,
                  const u64 *__restrict__ slice_dst, const u64 *__restrict__ slice_base, const u32 *__restrict__ slice_bucket,
                  u32 we, u32 *__restrict__ edges, uint8_t *__restrict__ aux, u64 capacity, const u32 *err_flag,
                  u64 *n_solid_out) {
  const u32 lane = threadIdx.x & 31;
  // a sub-range that could not be split any further (cannot happen for 42-bit remainders) must never pass silently:
  // the caller sees an impossible solid count
  if (blockIdx.x == 0 && threadIdx.x == 0 && *err_flag) *n_solid_out = ~0ull;
  const u64 n_slices = *n_slices_dev;
  for (u64 sl = (u64)blockIdx.x * 8 + (threadIdx.x >> 5); sl < n_slices; sl += (u64)gridDim.x * 8) {
    const u32 cnt = slice_count[sl];
    if (!cnt) continue;
    const u64 base = slice_base[sl], off = slice_dst[sl], b = slice_bucket[sl];
    for (u32 x = lane; x < cnt; x += 32) {
      if (off + x >= capacity) break;
      const u64 ent = list[base + x];
      const u64 key = (b << 48) | ((ent >> 22) << 6);
      u32 *e = edges + (off + x) * we;
      e[0] = (u32)(key >> 32);
      e[1] = (u32)key;
      if (we == 3) e[2] = 0;
      e[we - 1] |= (u32)(ent >> 6) & 0xFFFFu;
      aux[off + x] = (uint8_t)(ent & 3u);
    }
  }
}

int scan_counts(cudaStream_t st, const u32 *in, u64 n, u64 *out, u64 *total_dev, u64 *bsum) {
  const u64 nb = (n + kScanTile - 1) / kScanTile;
  k_scan32_sums<<<(unsigned)nb, kScanThreads, 0, st>>>(in, n, bsum);
  CK_LAUNCH();
  k_scan_u64<<<1, 1024, 0, st>>>(bsum, nb, total_dev);
  CK_LAUNCH();
  k_scan32_apply<<<(unsigned)nb, kScanThreads, 0, st>>>(in, n, bsum, out);
  CK_LAUNCH();
  return MHB_OK;
}

template <class G>
static int launch_hash_count(cudaStream_t st, const uint2 *recs, const u64 *slice_start, const u64 *n_slices_dev, int m,
                             u32 *misc, u64 *list, u32 *slice_count, u64 *mul_hist) {
  static int bps = 0;
  const size_t smem = sizeof(HcShared<G>);
  if (!bps) {
    CK(cudaFuncSetAttribute(k_hash_count<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_hash_count<G>, G::THREADS, smem));
    if (bps < 1) return mhb_set_error(MHB_ERR_CUDA, "hash-count kernel does not fit an SM (%zu B shared memory)", smem);
    if (getenv("MHB_VERBOSE")) fprintf(stderr, "[mhb] hash count: %d threads, %d slots, %zu B smem, %d CTA/SM, slice %u\n", G::THREADS, G::SLOTS, smem, bps, G::SLICE);
  }
  k_hash_count<G><<<sm_count() * bps, G::THREADS, smem, st>>>(recs, slice_start, n_slices_dev, m, misc, list, slice_count,
                                                             mul_hist, misc + 1);
  CK_LAUNCH();
  return MHB_OK;
}

struct HcLayout {
  size_t sort_ws, off_bounds, off_bcnt, off_soff, off_bsum, off_misc, off_scount, off_sdst, off_sbase, off_sbucket, off_sstart,
      off_list, total;
  uint64_t max_slices;
};
HcLayout hc_layout(uint64_t n, int32_t m) {
  HcLayout L;
  auto pad = [](size_t x) { return (x + 255) & ~(size_t)255; };
  L.max_slices = n / HcGeomB::SLICE + 65536 + 2;  // every bucket has ceil(records / SLICE) slices
  L.sort_ws = pad(mhb_sort_workspace_bytes(n, 2));
  size_t p = L.sort_ws;
  L.off_bounds = p;
  p += pad(65537 * 8);
  L.off_bcnt = p;
  p += pad(65537 * 4);
  L.off_soff = p;
  p += pad(65537 * 8);
  L.off_bsum = p;
  p += pad((L.max_slices / kScanTile + 4) * 8);
  L.off_misc = p;
  p += 256;
  L.off_scount = p;
  p += pad(L.max_slices * 4);
  L.off_sdst = p;
  p += pad(L.max_slices * 8);
  L.off_sbase = p;
  p += pad(L.max_slices * 8);
  L.off_sbucket = p;
  p += pad(L.max_slices * 4);
  L.off_sstart = p;
  p += pad((L.max_slices + 1) * 8);
  L.off_list = p;
  p += pad((size_t)(n / (uint64_t)(m < 1 ? 1 : m) + L.max_slices + 8) * 8);
  L.total = p;
  return L;
}

}  // namespace

extern "C" int mhb_count_hashed_supported(uint32_t k, int32_t m) {
  return count_record_words(k) == 2 && 2 * (k + 1) >= 24 && m >= 1 && m <= kHcHist;
}

extern "C" size_t mhb_count_hashed_workspace_bytes(uint64_t n, uint32_t k, int32_t m) {
  (void)k;
  return hc_layout(n, m).total;
}

extern "C" int mhb_count_solid_hashed(void *stream, uint32_t *recs_a, uint32_t *recs_b, uint64_t n, uint32_t k, int32_t m,
                                      const uint64_t *hist_byte5, uint32_t *edges_out, uint8_t *aux_out,
                                      uint64_t capacity_edges, uint64_t *mul_hist, uint64_t *n_solid_out, void *ws,
                                      size_t ws_bytes) {
  if (!mhb_count_hashed_supported(k, m)) return mhb_set_error(MHB_ERR_ARG, "hashed count needs 8-byte records (11 <= k <= 28) and 1 <= m <= %d", kHcHist);
  if (!mul_hist || !n_solid_out || !ws) return mhb_set_error(MHB_ERR_ARG, "bad args");
  if (n == 0) return MHB_OK;
  if (n >= (1ull << 40)) return mhb_set_error(MHB_ERR_ARG, "too many records for one hashed count call");
  const HcLayout L = hc_layout(n, m);
  if (ws_bytes < L.total) return mhb_set_error(MHB_ERR_ARG, "hashed count workspace too small (%zu < %zu)", ws_bytes, L.total);
  cudaStream_t st = (cudaStream_t)stream;
  // 1. group by the leading 24 key bits: stable passes on key bytes 5, 6, 7
  const uint8_t bytes[3] = {5, 6, 7};
  int in_b = 0;
  if (int rc = mhb_sort_records_impl(st, recs_a, recs_b, n, 2, bytes, 3, hist_byte5, ws, L.sort_ws, &in_b, nullptr)) return rc;
  const uint2 *recs = (const uint2 *)(in_b ? recs_b : recs_a);
  char *w = (char *)ws;
  u64 *bounds = (u64 *)(w + L.off_bounds);
  u32 *bcnt = (u32 *)(w + L.off_bcnt);
  u64 *slice_off = (u64 *)(w + L.off_soff);
  u64 *bsum = (u64 *)(w + L.off_bsum);
  u32 *misc = (u32 *)(w + L.off_misc);  // [0] ticket, [1] error flag, [2..3] number of slices (u64)
  u32 *slice_count = (u32 *)(w + L.off_scount);
  u64 *slice_dst = (u64 *)(w + L.off_sdst);
  u64 *slice_base = (u64 *)(w + L.off_sbase);
  u32 *slice_bucket = (u32 *)(w + L.off_sbucket);
  u64 *slice_start = (u64 *)(w + L.off_sstart);
  u64 *list = (u64 *)(w + L.off_list);
  u64 *n_slices_dev = (u64 *)(misc + 2);
  CK(cudaMemsetAsync(misc, 0, 256, st));
  CK(cudaMemsetAsync(slice_count, 0, L.max_slices * 4, st));
  // 2. bucket boundaries, slices per bucket
  k_bucket_bounds<<<(65537 + 255) / 256, 256, 0, st>>>(recs, n, bounds);
  CK_LAUNCH();
  k_slice_counts<<<65536 / 256, 256, 0, st>>>(bounds, HcGeomB::SLICE, bcnt);
  CK_LAUNCH();
  if (int rc = scan_counts(st, bcnt, 65536, slice_off, n_slices_dev, bsum)) return rc;
  CK(cudaMemcpyAsync(slice_off + 65536, n_slices_dev, 8, cudaMemcpyDeviceToDevice, st));
  k_slice_table<<<(unsigned)((L.max_slices + 1 + 255) / 256), 256, 0, st>>>(recs, bounds, slice_off, n_slices_dev, n, m, slice_start,
                                                                            slice_base, slice_bucket);
  CK_LAUNCH();
  // 3. per-slice hash aggregation
  if (int rc = launch_hash_count<HcGeomB>(st, recs, slice_start, n_slices_dev, m, misc, list, slice_count, mul_hist)) return rc;
  // 4. offsets + edges (the scan runs over the allocated maximum; unused slice ids hold zero)
  if (int rc = scan_counts(st, slice_count, L.max_slices, slice_dst, n_solid_out, bsum)) return rc;
  k_hash_gather<<<sm_count() * 4, 256, 0, st>>>(list, n_slices_dev, slice_count, slice_dst, slice_base, slice_bucket,
                                               words_per_edge(k), edges_out, aux_out, capacity_edges, misc + 1, n_solid_out);
  CK_LAUNCH();
  return MHB_OK;
}
