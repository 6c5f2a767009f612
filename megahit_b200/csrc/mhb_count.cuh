// mhb_count.cuh -- `count` stage kernels: edge extraction, solid-edge counting, mercy bookkeeping.
// Reference: voutcn/megahit src/sorting/kmer_counter.cpp (line numbers cited per kernel).
#pragma once
#include "mhb.h"
#include "mhb_kernels.cuh"

namespace mhb {

// ------------------------------------------------------------------------------------------------
// Streaming reads through shared memory with 1-D TMA (cp.async.bulk + mbarrier), two stages.
// A CTA walks batches of kReadsPerBatch consecutive reads (static round-robin over the grid); warp w
// handles reads w, w+NW, ... of the batch and calls f(read_id, s, nwords, L) with s pointing at the
// read's packed words (shared memory, or global memory for batches that do not fit a stage).
// ------------------------------------------------------------------------------------------------
static constexpr int kReadsPerBatch = 64;
static constexpr int kStageWords = 4096;  // 16 KiB per stage
static constexpr int kExtractThreads = 256;

struct ReadsView {
  const u32 *bin;
  u64 bin_words;
  u64 n_reads;
  u32 fixed_len;
  u32 fixed_stride;  // 1 + ceil(fixed_len/16)
  const u64 *rec_off;
  const u64 *edge_off;
  __device__ __forceinline__ u64 rec_start(u64 r) const { return fixed_len ? r * fixed_stride : rec_off[r]; }
};

template <class F>
__device__ __forceinline__ void for_each_read(const ReadsView &rv, F &&f) {
  __shared__ __align__(16) u32 s_stage[2][kStageWords];
  __shared__ __align__(8) u64 s_bar[2];
  const u32 tid = threadIdx.x, warp = tid >> 5;
  constexpr int NW = kExtractThreads / 32;
  const u64 n_batches = (rv.n_reads + kReadsPerBatch - 1) / kReadsPerBatch;
  if (tid == 0) {
    mbar_init(&s_bar[0], 1);
    mbar_init(&s_bar[1], 1);
    mbar_fence_init();
  }
  __syncthreads();

  // geometry of a batch: [a0, a1) = 16-byte aligned word range holding its records
  auto geom = [&](u64 b, u64 &r0, u64 &r1, u64 &a0, u64 &a1) {
    r0 = b * kReadsPerBatch;
    r1 = r0 + kReadsPerBatch < rv.n_reads ? r0 + kReadsPerBatch : rv.n_reads;
    const u64 w0 = rv.rec_start(r0);
    const u64 w1 = r1 < rv.n_reads ? rv.rec_start(r1) : rv.bin_words;
    a0 = w0 & ~3ull;
    a1 = (w1 + 3) & ~3ull;
  };
  auto issue = [&](u64 b, int st) {
    u64 r0, r1, a0, a1;
    geom(b, r0, r1, a0, a1);
    if (a1 - a0 <= (u64)kStageWords && tid == 0) {
      const u32 bytes = (u32)(a1 - a0) * 4;
      mbar_expect_tx(&s_bar[st], bytes);
      bulk_g2s(&s_stage[st][0], rv.bin + a0, bytes, &s_bar[st]);
    }
  };

  u32 parity[2] = {0, 0};
  u64 b = blockIdx.x;
  int st = 0;
  if (b < n_batches) issue(b, 0);
  for (; b < n_batches; b += gridDim.x, st ^= 1) {
    const u64 nb = b + gridDim.x;
    if (nb < n_batches) issue(nb, st ^ 1);  // stage st^1 was released by the __syncthreads below
    u64 r0, r1, a0, a1;
    geom(b, r0, r1, a0, a1);
    const bool staged = (a1 - a0) <= (u64)kStageWords;
    if (staged) {
      mbar_wait(&s_bar[st], parity[st]);
      parity[st] ^= 1;
    }
    for (u64 r = r0 + warp; r < r1; r += NW) {
      const u64 w = rv.rec_start(r);
      const u32 *rec = staged ? &s_stage[st][w - a0] : rv.bin + w;
      const u32 L = rec[0];
      f(r, rec + 1, div_ceil(L, 16), L);
    }
    __syncthreads();  // everyone is done with stage st before it is refilled
  }
}

// ------------------------------------------------------------------------------------------------
// K-extract (A1-A3; kmer_counter.cpp:114-252): one record per (k+1)-mer occurrence.
// ------------------------------------------------------------------------------------------------
template <int W, int WR>
__global__ void __launch_bounds__(kExtractThreads)
    k_count_extract(ReadsView rv, u32 k, u32 *__restrict__ records, u64 *hist, int hist_byte) {
  __shared__ u32 s_hist[256];
  for (int i = threadIdx.x; i < 256; i += kExtractThreads) s_hist[i] = 0;
  const u32 lane = lane_id();
  const u32 K1 = k + 1;
  for_each_read(rv, [&](u64 r, const u32 *s, u32 nwords, u32 L) {
    if (L < K1) return;  // kmer_counter.cpp:124
    const u32 n_e = L - k;
    const u64 base = rv.fixed_len ? r * (u64)(rv.fixed_len - k) : rv.edge_off[r];
    for (u32 q0 = 0; q0 < n_e; q0 += 32) {
      const u32 q = q0 + lane;
      if (q < n_e) {
        u32 rec[WR], strand;
        make_count_record<W, WR>(s, nwords, L, k, q, rec, strand);
        st_rec<WR>(records, base + q, rec);
        if (hist) atomicAdd(&s_hist[rec_byte<WR>(rec, hist_byte)], 1u);
      }
    }
  });
  __syncthreads();
  if (hist)
    for (int i = threadIdx.x; i < 256; i += kExtractThreads)
      if (s_hist[i]) atomicAdd((unsigned long long *)&hist[i], (unsigned long long)s_hist[i]);
}

// ------------------------------------------------------------------------------------------------
// K-extract restricted to a range of leading bytes (A13; base_engine.cpp:254-281 Lv1 passes over bucket ranges):
// when the records of a whole library do not fit in HBM the count stage runs in rounds, each round extracting only
// the edges whose first eight bases (the 16-bit bucket id) lie in [lo, hi].  Two launches, no atomics, read order kept:
//   WRITE = false: per_read[r] = number of in-range edges of read r (+ optional histogram of record byte hist_byte)
//   WRITE = true : per_read[r] = exclusive prefix of those counts; in-range records are stored compactly from there
// ------------------------------------------------------------------------------------------------
template <int W, int WR, bool WRITE>
__global__ void __launch_bounds__(kExtractThreads)
    k_count_extract_range(ReadsView rv, u32 k, u32 lo, u32 hi, u64 *__restrict__ per_read, u32 *__restrict__ records,
                          u64 *hist, int hist_byte) {
  __shared__ u32 s_hist[256];
  for (int i = threadIdx.x; i < 256; i += kExtractThreads) s_hist[i] = 0;
  const u32 lane = lane_id();
  const u32 lt_mask = lanemask_lt();
  const u32 K1 = k + 1;
  for_each_read(rv, [&](u64 r, const u32 *s, u32 nwords, u32 L) {
    if (L < K1) {  // kmer_counter.cpp:124
      if (!WRITE && lane == 0) per_read[r] = 0;
      return;
    }
    const u32 n_e = L - k;
    u64 run = WRITE ? per_read[r] : 0ull;
    for (u32 q0 = 0; q0 < n_e; q0 += 32) {
      const u32 q = q0 + lane;
      u32 rec[WR], strand;
      bool in = false;
      if (q < n_e) {
        make_count_record<W, WR>(s, nwords, L, k, q, rec, strand);
        const u32 top = rec[0] >> 16;  // the 8-base bucket id (base_engine.h kNumBuckets)
        in = top >= lo && top <= hi;
      }
      const u32 mask = __ballot_sync(0xffffffffu, in);
      if (in) {
        if constexpr (WRITE) st_rec<WR>(records, run + __popc(mask & lt_mask), rec);
        if (hist) atomicAdd(&s_hist[rec_byte<WR>(rec, hist_byte)], 1u);
      }
      run += __popc(mask);
    }
    if (!WRITE && lane == 0) per_read[r] = run;
  });
  __syncthreads();
  if (hist)
    for (int i = threadIdx.x; i < 256; i += kExtractThreads)
      if (s_hist[i]) atomicAdd((unsigned long long *)&hist[i], (unsigned long long)s_hist[i]);
}

// ------------------------------------------------------------------------------------------------
// K-count helpers (A5/A6; kmer_counter.cpp:254-381)
// ------------------------------------------------------------------------------------------------
template <int WR>
__device__ __forceinline__ bool same_edge(const u32 (&a)[WR], const u32 (&b)[WR]) {
  bool eq = true;
#pragma unroll
  for (int j = 0; j < WR; ++j) {
    const u32 m = (j == WR - 1) ? ~63u : ~0u;
    eq = eq && ((a[j] & m) == (b[j] & m));
  }
  return eq;
}

static constexpr int kMulHistSmem = 1024;

// in-place exclusive scan of nb u64 values by ONE block; writes the grand total
static __global__ void __launch_bounds__(1024) k_scan_u64(u64 *v, u64 nb, u64 *total_out) {
  __shared__ u64 s_w[33];
  __shared__ u64 s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const u32 lane = lane_id(), warp = threadIdx.x >> 5;
  for (u64 base = 0; base < nb; base += 1024) {
    const u64 i = base + threadIdx.x;
    const u64 x = i < nb ? v[i] : 0;
    u64 inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      u64 t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= (u32)d) inc += t;
    }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      u64 w = s_w[lane], winc = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        u64 t = __shfl_up_sync(0xffffffffu, winc, d);
        if (lane >= (u32)d) winc += t;
      }
      s_w[lane] = winc - w;
      if (lane == 31) s_w[32] = winc;
    }
    __syncthreads();
    if (i < nb) v[i] = s_carry + s_w[warp] + inc - x;
    __syncthreads();
    if (threadIdx.x == 0) s_carry += s_w[32];
    __syncthreads();
  }
  if (threadIdx.x == 0 && total_out) *total_out = s_carry;
}

// ------------------------------------------------------------------------------------------------
// tip set: the solid edges that lack an incoming or outgoing solid neighbour (aux != 0), as
//   u64 capacity (power of two), u64 filter_words (power of two),
//   u32 filter[filter_words]           one-bit-per-hash prefilter (~32 bits per tip edge, L2 resident)
//   u32 table[capacity][1 + W]         open addressing: flags (0 = empty) followed by the (k+1)-mer
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline u64 tipset_capacity(u64 n_tip) {
  u64 c = 1024;
  while (c < 2 * n_tip) c <<= 1;
  return c;
}
__host__ __device__ inline u64 tipset_filter_words(u64 n_tip) {
  u64 c = 1024;
  while (c < n_tip) c <<= 1;
  return c;
}

template <int W>
__device__ __forceinline__ u32 hash_key(const u32 (&key)[W]) {
  u32 h = 0x9E3779B1u;
#pragma unroll
  for (int j = 0; j < W; ++j) {
    h = (h ^ key[j]) * 0x85EBCA77u;
    h ^= h >> 15;
  }
  h *= 0x2C1B3C6Du;
  return h ^ (h >> 13);
}
__device__ __forceinline__ u32 hash2(u32 h) {  // second, independent-ish hash for the bit filter
  h *= 0xC2B2AE3Du;
  return h ^ (h >> 16);
}

static __global__ void k_count_tips(const uint8_t *aux, u64 n, unsigned long long *out) {
  u64 c = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
    c += aux[i] != 0;
  for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
  if (lane_id() == 0 && c) atomicAdd(out, (unsigned long long)c);
}

template <int W>
__global__ void k_tipset_insert(const u32 *__restrict__ edges, const uint8_t *__restrict__ aux, u64 n, u32 k,
                                u32 *filter, u64 filter_words, u32 *table, u64 cap) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || aux[i] == 0) return;
  const u32 WE = words_per_edge(k);
  u32 key[W];
#pragma unroll
  for (int j = 0; j < W; ++j) {
    const u32 keep = 2 * (k + 1) - 32 * j;
    key[j] = edges[i * WE + j] & top_mask(keep > 32 ? 32 : keep);
  }
  const u32 h = hash_key<W>(key);
  const u32 fb = hash2(h) & (u32)(filter_words * 32 - 1);
  atomicOr(&filter[fb >> 5], 1u << (fb & 31));
  u64 slot = h & (cap - 1);
  while (true) {
    u32 *e = table + slot * (W + 1);
    if (atomicCAS(e, 0u, (u32)aux[i]) == 0u) {
#pragma unroll
      for (int j = 0; j < W; ++j) e[1 + j] = key[j];
      return;
    }
    slot = (slot + 1) & (cap - 1);
  }
}

// K-mercy (kmer_counter.cpp:307-367): per read min/max over the occurrences of tip edges.
// One warp per read, straight from global memory (the library is ~3 % of the count stage's traffic and
// L1 serves the re-reads), kMercyUnroll positions per lane per round so that the bit-filter probes of a
// whole 150 bp read are in flight together; the kernel is bound by L2 latency, not bandwidth.
static constexpr int kMercyUnroll = 4;

template <int W, int WR>
__global__ void __launch_bounds__(256)
    k_mark_mercy(ReadsView rv, u32 k, const u32 *__restrict__ filter, u64 filter_words, const u32 *__restrict__ table,
                 u64 cap, u32 *first_0_out, u32 *last_0_in) {
  const u32 lane = lane_id();
  const u32 K1 = k + 1;
  const u32 fmask = (u32)(filter_words * 32 - 1);
  for (u64 r = (u64)blockIdx.x * 8 + (threadIdx.x >> 5); r < rv.n_reads; r += (u64)gridDim.x * 8) {
    const u32 *rec0 = rv.bin + rv.rec_start(r);
    const u32 L = rec0[0];
    const u32 *s = rec0 + 1;
    const u32 nwords = div_ceil(L, 16);
    u32 first = 0xFFFFFFFFu;
    long long last = -1;
    if (L >= K1) {
      const u32 n_e = L - k;
      for (u32 q0 = 0; q0 < n_e; q0 += 32 * kMercyUnroll) {
        u32 key[kMercyUnroll][W], strand[kMercyUnroll], fw[kMercyUnroll], h[kMercyUnroll];
        bool live[kMercyUnroll];
#pragma unroll
        for (int u = 0; u < kMercyUnroll; ++u) {
          const u32 q = q0 + 32 * u + lane;
          live[u] = q < n_e;
          h[u] = 0;
          fw[u] = 0;
          strand[u] = 0;
          if (live[u]) {
            u32 rec[WR];
            make_count_record<W, WR>(s, nwords, L, k, q, rec, strand[u]);
#pragma unroll
            for (int j = 0; j < W; ++j) {
              const u32 keep = 2 * K1 - 32 * j;
              key[u][j] = rec[j] & top_mask(keep > 32 ? 32 : keep);
            }
            h[u] = hash_key<W>(key[u]);
            fw[u] = filter[(hash2(h[u]) & fmask) >> 5];
          }
        }
#pragma unroll
        for (int u = 0; u < kMercyUnroll; ++u) {
          if (!live[u] || !((fw[u] >> (hash2(h[u]) & 31)) & 1u)) continue;
          u64 slot = h[u] & (cap - 1);
          u32 flags = 0;
          while (true) {
            const u32 *e = table + slot * (W + 1);
            const u32 f = e[0];
            if (f == 0) break;
            bool eq = true;
#pragma unroll
            for (int j = 0; j < W; ++j) eq = eq && e[1 + j] == key[u][j];
            if (eq) {
              flags = f;
              break;
            }
            slot = (slot + 1) & (cap - 1);
          }
          if (flags) {
            const u32 off = L - K1 - (q0 + 32 * u + lane);  // offset in the reversed (package) read
            // no in, strand 0 -> last; no in, strand 1 -> first; no out, strand 0 -> first; no out, strand 1 -> last
            const bool to_last = ((flags & 1u) && strand[u] == 0) || ((flags & 2u) && strand[u] == 1);
            const bool to_first = ((flags & 1u) && strand[u] == 1) || ((flags & 2u) && strand[u] == 0);
            if (to_last) last = last > (long long)off ? last : (long long)off;
            if (to_first) first = first < off + 1 ? first : off + 1;
          }
        }
      }
    }
    for (int d = 16; d; d >>= 1) {
      const u32 f2 = __shfl_xor_sync(0xffffffffu, first, d);
      const long long l2 = __shfl_xor_sync(0xffffffffu, last, d);
      first = first < f2 ? first : f2;
      last = last > l2 ? last : l2;
    }
    if (lane == 0) {
      first_0_out[r] = first;
      last_0_in[r] = last < 0 ? 0xFFFFFFFFu : (u32)last;
    }
  }
}

// Rolling variant of k_mark_mercy for 8-byte records: a lane re-derives four consecutive canonical (k+1)-mers with
// make_count_records_roll (~55 instead of ~120 thread-instructions per record) and probes the filter for all four at once.
static __global__ void __launch_bounds__(256)
    k_mark_mercy_roll(ReadsView rv, u32 k, const u32 *__restrict__ filter, u64 filter_words, const u32 *__restrict__ table,
                      u64 cap, u32 *first_0_out, u32 *last_0_in) {
  constexpr int W = 2;
  const u32 lane = lane_id();
  const u32 K1 = k + 1;
  const u32 fmask = (u32)(filter_words * 32 - 1);
  for (u64 r = (u64)blockIdx.x * 8 + (threadIdx.x >> 5); r < rv.n_reads; r += (u64)gridDim.x * 8) {
    const u32 *rec0 = rv.bin + rv.rec_start(r);
    const u32 L = rec0[0];
    const u32 *s = rec0 + 1;
    const u32 nwords = div_ceil(L, 16);
    u32 first = 0xFFFFFFFFu;
    long long last = -1;
    if (L >= K1) {
      const u32 n_e = L - k;
      for (u32 q0 = 0; q0 < n_e; q0 += 128) {
        const u32 q = q0 + 4 * lane;
        u32 key[4][W], strand[4] = {0, 0, 0, 0}, fw[4] = {0, 0, 0, 0}, h[4] = {0, 0, 0, 0};
        bool live[4] = {false, false, false, false};
        if (q < n_e) {
          u64 rec[4];
          make_count_records_roll<4>(s, nwords, L, k, q, rec, strand);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            live[u] = q + u < n_e;
            key[u][0] = (u32)(rec[u] >> 32);
            key[u][1] = (u32)rec[u] & ~63u;  // drop prev/next: the (k+1)-mer alone, as the tip set stores it
            if (live[u]) {
              h[u] = hash_key<W>(key[u]);
              fw[u] = filter[(hash2(h[u]) & fmask) >> 5];
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (!live[u] || !((fw[u] >> (hash2(h[u]) & 31)) & 1u)) continue;
          u64 slot = h[u] & (cap - 1);
          u32 flags = 0;
          while (true) {
            const u32 *e = table + slot * (W + 1);
            const u32 f = e[0];
            if (f == 0) break;
            if (e[1] == key[u][0] && e[2] == key[u][1]) {
              flags = f;
              break;
            }
            slot = (slot + 1) & (cap - 1);
          }
          if (flags) {
            const u32 off = L - K1 - (q + u);  // offset in the reversed (package) read
            const bool to_last = ((flags & 1u) && strand[u] == 0) || ((flags & 2u) && strand[u] == 1);
            const bool to_first = ((flags & 1u) && strand[u] == 1) || ((flags & 2u) && strand[u] == 0);
            if (to_last) last = last > (long long)off ? last : (long long)off;
            if (to_first) first = first < off + 1 ? first : off + 1;
          }
        }
      }
    }
    for (int d = 16; d; d >>= 1) {
      const u32 f2 = __shfl_xor_sync(0xffffffffu, first, d);
      const long long l2 = __shfl_xor_sync(0xffffffffu, last, d);
      first = first < f2 ? first : f2;
      last = last > l2 ? last : l2;
    }
    if (lane == 0) {
      first_0_out[r] = first;
      last_0_in[r] = last < 0 ? 0xFFFFFFFFu : (u32)last;
    }
  }
}


}  // namespace mhb

namespace mhb {

// ------------------------------------------------------------------------------------------------
// K-count v3 (A5/A6): one pass, each LANE walks IPL consecutive sorted records.
//
// A warp claims a chunk of 32*IPL records by ticket and stages it in shared memory (coalesced loads,
// lane-blocked conflict-free layout).  Every lane scans its IPL records once, keeping byte-packed
// prev/next tallies (kmer_counter.cpp:279-295) for the run it is in; runs that start and end inside a
// lane are judged on the spot, the piece before a lane's first run head ("front") and the piece after
// its last head ("back") are stitched across lanes by one segmented warp scan, and the chunk's last run
// is followed past the chunk end with ballots.  A run is OWNED by the lane holding its first record, so
// solid edges come out in sorted order.  No serial dependency between chunks: the judge kernel leaves each
// chunk's solid runs as a compact list (slot, judged word) in a scratch area plus the chunk's total; a
// three-phase scan turns the totals into output offsets; k_count_write then gathers the keys and packs the
// edges (PackEdge, kmer_counter.cpp:32-52).  (A decoupled look-back over 512-record chunks was measured to
// spend > 55 % of the kernel waiting on the chunk chain.)
// ------------------------------------------------------------------------------------------------
static constexpr int kCount3Warps = 8;
__host__ __device__ constexpr int count3_ipl(int wr) { return wr <= 4 ? 16 : (wr <= 8 ? 8 : 4); }
__host__ __device__ constexpr int count3_lane_stride(int wr) {  // words; padded against bank conflicts
  return count3_ipl(wr) * wr + (wr == 2 ? 2 : (wr == 4 ? 4 : ((count3_ipl(wr) * wr) % 2 == 0 ? 1 : 0)));
}
__host__ __device__ constexpr int count3_warp_words(int wr) {
  return 32 * count3_lane_stride(wr) + ((wr + 3) & ~3) /*record a-1*/ + 32 * count3_ipl(wr) /*info*/;
}

__device__ __forceinline__ u64 spread16(u64 packed8) {  // 4 byte counters -> 4 u16 fields
  return (packed8 & 0xFFull) | ((packed8 & 0xFF00ull) << 8) | ((packed8 & 0xFF0000ull) << 16) |
         ((packed8 & 0xFF000000ull) << 24);
}

struct Tally {  // count + 4 prev + 4 next tallies as 16-bit fields
  u32 cnt;
  u64 p, n;
};

template <int WR>
__global__ void __launch_bounds__(kCount3Warps * 32)
    k_count_lanes(const u32 *__restrict__ recs, u64 n, u32 k, int m, u32 n_chunks, u32 *ticket,
                  uint2 *__restrict__ solid_list /*n entries: chunk c owns [c*CH, (c+1)*CH)*/,
                  u32 *__restrict__ chunk_count, u64 *mul_hist) {
  constexpr int IPL = count3_ipl(WR), CH = 32 * IPL, LS = count3_lane_stride(WR);
  extern __shared__ __align__(16) u32 smem_w[];
  __shared__ u32 s_hist[kMulHistSmem];
  const u32 lane = lane_id(), warp = threadIdx.x >> 5;
  u32 *s_rec = smem_w + (size_t)warp * count3_warp_words(WR);  // lane-blocked records
  u32 *s_prev = s_rec + 32 * LS;                                // record a-1
  u32 *s_info = s_prev + ((WR + 3) & ~3);                       // per owned run head: judged result
  (void)k;
  for (int i = threadIdx.x; i < kMulHistSmem; i += kCount3Warps * 32) s_hist[i] = 0;
  __syncthreads();
  u32 n_ones = 0;

  auto judge = [&](u32 cnt, const u32 (&tp)[4], const u32 (&tn)[4]) -> u32 {
    // -> 1 | solid<<1 | no_in<<2 | no_out<<3 | min(cnt,65535)<<8 ; also feeds the multiplicity histogram
    const u32 c16 = cnt > 65535u ? 65535u : cnt;
    if (c16 == 1u) ++n_ones;
    else if (c16 < (u32)kMulHistSmem) atomicAdd(&s_hist[c16], 1u);
    else atomicAdd((unsigned long long *)&mul_hist[c16], 1ull);
    u32 word = 1u | (c16 << 8);
    if ((long long)cnt >= (long long)m) {
      bool has_in = false, has_out = false;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        has_in = has_in || (long long)tp[c] >= (long long)m;
        has_out = has_out || (long long)tn[c] >= (long long)m;
      }
      word |= 2u | (has_in ? 0u : 4u) | (has_out ? 0u : 8u);
    }
    return word;
  };

  while (true) {
    u32 chunk = 0;
    if (lane == 0) chunk = atomicAdd(ticket, 1u);
    chunk = __shfl_sync(0xffffffffu, chunk, 0);
    if (chunk >= n_chunks) break;
    const u64 a = (u64)chunk * CH;
    const u64 b = a + CH < n ? a + CH : n;
    const u32 n_here = (u32)(b - a);

    // ---- stage the chunk: coalesced global reads -> lane-blocked shared layout ----
#pragma unroll
    for (int i = 0; i < IPL; ++i) {
      const u32 t = (u32)i * 32 + lane;
      if (t < n_here) {
        u32 r[WR];
        ld_rec<WR>(recs, a + t, r);
        u32 *dst = s_rec + (t / IPL) * LS + (t % IPL) * WR;
        if constexpr (WR == 2) *reinterpret_cast<uint2 *>(dst) = make_uint2(r[0], r[1]);
        else if constexpr (WR == 4) *reinterpret_cast<uint4 *>(dst) = make_uint4(r[0], r[1], r[2], r[3]);
        else {
#pragma unroll
          for (int j = 0; j < WR; ++j) dst[j] = r[j];
        }
      }
    }
    if (lane < WR) s_prev[lane] = a > 0 ? recs[(a - 1) * WR + lane] : 0u;
    __syncwarp();

    // ---- every lane walks its records ----
    const u32 my_first = lane * IPL;
    const u32 my_n = n_here > my_first ? (n_here - my_first < (u32)IPL ? n_here - my_first : (u32)IPL) : 0u;
    u32 prev[WR];
    {
      const u32 *pp = lane == 0 ? s_prev : s_rec + (lane - 1) * LS + (IPL - 1) * WR;
#pragma unroll
      for (int j = 0; j < WR; ++j) prev[j] = pp[j];
    }
    u32 cnt = 0, f_cnt = 0, head_slot = 0, solid_mask = 0, n_solid_lane = 0;
    u64 cp = 0, cn = 0, f_cp = 0, f_cn = 0;  // byte-packed tallies (<= 16 per lane), byte 4 = sentinel
    bool seen_head = false;
    const u32 *mine = s_rec + lane * LS;
    for (u32 j = 0; j < my_n; ++j) {
      u32 r[WR];
      if constexpr (WR == 2) {
        const uint2 v = *reinterpret_cast<const uint2 *>(mine + j * 2);
        r[0] = v.x;
        r[1] = v.y;
      } else if constexpr (WR == 4) {
        const uint4 v = *reinterpret_cast<const uint4 *>(mine + j * 4);
        r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
      } else {
#pragma unroll
        for (int q = 0; q < WR; ++q) r[q] = mine[j * WR + q];
      }
      const bool head = (a + my_first + j == 0) || !same_edge<WR>(r, prev);
      if (head) {
        if (!seen_head) {
          f_cnt = cnt; f_cp = cp; f_cn = cn;
          seen_head = true;
        } else {  // a run that lives entirely inside this lane
          u32 tp[4], tn[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            tp[c] = (u32)(cp >> (8 * c)) & 0xFFu;
            tn[c] = (u32)(cn >> (8 * c)) & 0xFFu;
          }
          const u32 word = judge(cnt, tp, tn);
          s_info[my_first + head_slot] = word;
          if (word & 2u) {
            solid_mask |= 1u << head_slot;
            ++n_solid_lane;
          }
        }
        cnt = 0; cp = 0; cn = 0;
        head_slot = j;
      }
      const u32 pn = r[WR - 1] & 63u;
      ++cnt;
      cp += 1ull << (8 * (pn >> 3));
      cn += 1ull << (8 * (pn & 7u));
#pragma unroll
      for (int q = 0; q < WR; ++q) prev[q] = r[q];
    }
    if (!seen_head) {  // the whole lane is the middle of somebody else's run
      f_cnt = cnt; f_cp = cp; f_cn = cn;
    }

    // ---- stitch runs across lanes: S(y) = tallies of lanes y.. up to and including the first head lane ----
    Tally S = {f_cnt, spread16(f_cp), spread16(f_cn)};
    bool stop = seen_head;  // a head exists in [y, y+span)
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 o_cnt = __shfl_down_sync(0xffffffffu, S.cnt, d);
      const u64 o_p = __shfl_down_sync(0xffffffffu, S.p, d);
      const u64 o_n = __shfl_down_sync(0xffffffffu, S.n, d);
      const bool o_stop = __shfl_down_sync(0xffffffffu, (int)stop, d) != 0;
      if (lane + d < 32 && !stop) {
        S.cnt += o_cnt; S.p += o_p; S.n += o_n;
        stop = o_stop;
      }
    }
    Tally nxt;  // S(lane+1)
    nxt.cnt = __shfl_down_sync(0xffffffffu, S.cnt, 1);
    nxt.p = __shfl_down_sync(0xffffffffu, S.p, 1);
    nxt.n = __shfl_down_sync(0xffffffffu, S.n, 1);
    bool later_head = __shfl_down_sync(0xffffffffu, (int)stop, 1) != 0;
    if (lane == 31) {
      nxt.cnt = 0; nxt.p = 0; nxt.n = 0;
      later_head = false;
    }

    // ---- the chunk's last run may continue past the chunk: follow it (warp-cooperative) ----
    const u32 any_head = __ballot_sync(0xffffffffu, seen_head);
    u32 t_cnt = 0, t_p[4] = {0, 0, 0, 0}, t_n[4] = {0, 0, 0, 0};
    if (any_head && b < n) {
      u32 key[WR];
      {
        const u32 t = n_here - 1;
        const u32 *lp = s_rec + (t / IPL) * LS + (t % IPL) * WR;
#pragma unroll
        for (int j = 0; j < WR; ++j) key[j] = lp[j];
      }
      for (u64 pos = b; pos < n; pos += 32) {
        const u64 i = pos + lane;
        u32 r[WR];
        bool same = false;
        if (i < n) {
          ld_rec<WR>(recs, i, r);
          same = same_edge<WR>(r, key);
        } else {
#pragma unroll
          for (int j = 0; j < WR; ++j) r[j] = 0;
        }
        const u32 diff = ~__ballot_sync(0xffffffffu, same);
        const u32 seg = diff ? ((1u << (__ffs(diff) - 1)) - 1u) : 0xffffffffu;  // lanes still in the run
        const u32 pn = r[WR - 1] & 63u;
        t_cnt = min(t_cnt + (u32)__popc(seg), 0x40000000u);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          t_p[c] = min(t_p[c] + (u32)__popc(seg & __ballot_sync(0xffffffffu, (pn >> 3) == (u32)c)), 0x40000000u);
          t_n[c] = min(t_n[c] + (u32)__popc(seg & __ballot_sync(0xffffffffu, (pn & 7u) == (u32)c)), 0x40000000u);
        }
        if (diff) break;
      }
    }

    // ---- judge each lane's last run (the one that may span lanes) ----
    if (seen_head) {
      u32 tp[4], tn[4];
      const u64 bp = spread16(cp) + nxt.p, bn = spread16(cn) + nxt.n;
      u32 total = cnt + nxt.cnt;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        tp[c] = (u32)(bp >> (16 * c)) & 0xFFFFu;
        tn[c] = (u32)(bn >> (16 * c)) & 0xFFFFu;
      }
      if (!later_head) {  // this run reaches the end of the chunk: add what lies beyond
        total = min(total + t_cnt, 0x40000000u);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          tp[c] += t_p[c];
          tn[c] += t_n[c];
        }
      }
      const u32 word = judge(total, tp, tn);
      s_info[my_first + head_slot] = word;
      if (word & 2u) {
        solid_mask |= 1u << head_slot;
        ++n_solid_lane;
      }
    }

    // ---- leave this chunk's solid runs as a compact, ordered list ----
    u32 inc = n_solid_lane;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= (u32)d) inc += t;
    }
    if (lane == 31) chunk_count[chunk] = inc;
    u32 at = inc - n_solid_lane;
    while (solid_mask) {
      const u32 j = __ffs(solid_mask) - 1;
      solid_mask &= solid_mask - 1;
      solid_list[a + at] = make_uint2(my_first + j, s_info[my_first + j]);
      ++at;
    }
    __syncwarp();
  }

  if (n_ones) atomicAdd(&s_hist[1], n_ones);
  __syncthreads();
  for (int c = threadIdx.x; c < kMulHistSmem; c += kCount3Warps * 32)
    if (s_hist[c]) atomicAdd((unsigned long long *)&mul_hist[c], (unsigned long long)s_hist[c]);
}


// ---- three-phase exclusive scan of u32 counts into u64 offsets (4096 entries per block) ----
static constexpr int kScanThreads = 1024, kScanItems = 4, kScanTile = kScanThreads * kScanItems;

static __global__ void __launch_bounds__(kScanThreads) k_scan32_sums(const u32 *in, u64 n, u64 *bsum) {
  __shared__ u32 s_scan[kScanThreads / 32 + 1];
  const u64 base = (u64)blockIdx.x * kScanTile + (u64)threadIdx.x * kScanItems;
  u32 c = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j)
    if (base + j < n) c += in[base + j];
  u32 total;
  block_excl_scan<kScanThreads>(c, s_scan, total);
  if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

static __global__ void __launch_bounds__(kScanThreads) k_scan32_apply(const u32 *in, u64 n, const u64 *bsum, u64 *out) {
  __shared__ u32 s_scan[kScanThreads / 32 + 1];
  const u64 base = (u64)blockIdx.x * kScanTile + (u64)threadIdx.x * kScanItems;
  u32 v[kScanItems], c = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    v[j] = base + j < n ? in[base + j] : 0u;
    c += v[j];
  }
  u32 total;
  u64 off = bsum[blockIdx.x] + block_excl_scan<kScanThreads>(c, s_scan, total);
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    if (base + j < n) out[base + j] = off;
    off += v[j];
  }
}

// same three phases for u64 values, in place (exclusive)
static __global__ void __launch_bounds__(kScanThreads) k_scan64_sums(const u64 *in, u64 n, u64 *bsum) {
  __shared__ u64 s_w[33];
  const u64 base = (u64)blockIdx.x * kScanTile + (u64)threadIdx.x * kScanItems;
  u64 c = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j)
    if (base + j < n) c += in[base + j];
  for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
  if (lane_id() == 0) s_w[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x < 32) {
    u64 v = s_w[threadIdx.x];
    for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (threadIdx.x == 0) bsum[blockIdx.x] = v;
  }
}

static __global__ void __launch_bounds__(kScanThreads) k_scan64_apply(u64 *v, u64 n, const u64 *bsum) {
  __shared__ u64 s_w[33];
  const u32 lane = lane_id(), warp = threadIdx.x >> 5;
  const u64 base = (u64)blockIdx.x * kScanTile + (u64)threadIdx.x * kScanItems;
  u64 x[kScanItems], c = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    x[j] = base + j < n ? v[base + j] : 0ull;
    c += x[j];
  }
  u64 inc = c;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const u64 t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= (u32)d) inc += t;
  }
  if (lane == 31) s_w[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const u64 w = s_w[lane];
    u64 winc = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u64 t = __shfl_up_sync(0xffffffffu, winc, d);
      if (lane >= (u32)d) winc += t;
    }
    s_w[lane] = winc - w;
  }
  __syncthreads();
  u64 off = bsum[blockIdx.x] + s_w[warp] + inc - c;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    if (base + j < n) v[base + j] = off;
    off += x[j];
  }
}

// PackEdge (kmer_counter.cpp:32-52): one warp per chunk turns the chunk's solid list into edges
template <int WR>
__global__ void __launch_bounds__(256)
    k_count_write(const u32 *__restrict__ recs, u32 k, u32 n_chunks, const uint2 *__restrict__ solid_list,
                  const u32 *__restrict__ chunk_count, const u64 *__restrict__ chunk_off, u32 *__restrict__ edges,
                  uint8_t *__restrict__ aux, u64 capacity) {
  constexpr int CH = 32 * count3_ipl(WR);
  const u32 W = count_key_words(k), WE = words_per_edge(k);
  const u32 lane = lane_id();
  for (u64 chunk = (u64)blockIdx.x * 8 + (threadIdx.x >> 5); chunk < n_chunks; chunk += (u64)gridDim.x * 8) {
    const u32 cnt = chunk_count[chunk];
    const u64 off = chunk_off[chunk], a = chunk * CH;
    for (u32 x = lane; x < cnt; x += 32) {
      if (off + x >= capacity) break;
      const uint2 ent = solid_list[a + x];
      u32 r[WR];
      ld_rec<WR>(recs, a + ent.x, r);
      r[WR - 1] &= ~63u;
      u32 *e = edges + (off + x) * WE;
      for (u32 y = 0; y < WE; ++y) e[y] = (y < W && y < (u32)WR) ? pick<WR>(r, y) : 0u;
      e[WE - 1] |= ent.y >> 8;
      aux[off + x] = (uint8_t)((ent.y >> 2) & 3u);
    }
  }
}

}  // namespace mhb
