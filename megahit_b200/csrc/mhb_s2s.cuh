// mhb_s2s.cuh -- `seq2sdbg` stage kernels: item extraction and SdBG emission.
// Reference: voutcn/megahit src/sorting/seq_to_sdbg.cpp, src/sdbg/sdbg_writer.cpp.
#pragma once
#include "mhb.h"
#include "mhb_kernels.cuh"

namespace mhb {

struct SeqsView {
  const u32 *words;
  u64 n_words;
  u64 n_seqs;
  u32 fixed_len;
  const u64 *word_off;
  const u32 *len;
  const u64 *item_off;
  const uint16_t *mult;
  u32 fixed_stride;
};

// S-extract (A8/A9; seq_to_sdbg.cpp:530-700): thread t builds sort item t.
template <int W>
__global__ void __launch_bounds__(256)
    k_s2s_extract(SeqsView sv, u32 k, u32 *__restrict__ records, u64 n_items, u64 *hist, int hist_byte) {
  __shared__ u32 s_hist[256];
  for (int i = threadIdx.x; i < 256; i += 256) s_hist[i] = 0;
  __syncthreads();
  for (u64 t = (u64)blockIdx.x * 256 + threadIdx.x; t < n_items; t += (u64)gridDim.x * 256) {
    u64 seq, rem;
    u32 L;
    const u32 *s;
    u32 nwords;
    if (sv.fixed_len) {
      L = sv.fixed_len;
      const u64 ips = 2ull * (L - k + 2);
      seq = t / ips;
      rem = t - seq * ips;
      nwords = div_ceil(L, 16);
      s = sv.words + seq * (sv.fixed_stride ? sv.fixed_stride : nwords);
    } else {
      u64 lo = 0, hi = sv.n_seqs;  // last seq with item_off[seq] <= t
      while (hi - lo > 1) {
        const u64 mid = (lo + hi) >> 1;
        if (sv.item_off[mid] <= t) lo = mid; else hi = mid;
      }
      seq = lo;
      rem = t - sv.item_off[seq];
      L = sv.len[seq];
      nwords = div_ceil(L, 16);
      s = sv.words + sv.word_off[seq];
    }
    const u32 per_strand = L - k + 2;
    const u32 strand = rem >= per_strand ? 1u : 0u;
    const u32 offset = (u32)(rem - (u64)strand * per_strand);
    u32 rec[W];
    const u32 mult = sv.mult ? (u32)sv.mult[seq] : (s[sv.fixed_stride - 1] & 0xFFFFu);
    make_s2s_record<W>(s, nwords, L, k, strand, offset, mult, rec);
    st_rec<W>(records, t, rec);
    if (hist) atomicAdd(&s_hist[rec_byte<W>(rec, hist_byte)], 1u);
  }
  __syncthreads();
  if (hist)
    for (int i = threadIdx.x; i < 256; i += 256)
      if (s_hist[i]) atomicAdd((unsigned long long *)&hist[i], (unsigned long long)s_hist[i]);
}

// S-extract restricted to the items whose 16-bit bucket id (first eight bases) lies in [lo, hi] (A13: seq2sdbg in
// rounds when the items of all sequences do not fit in HBM; base_engine.cpp:254-281).  records == nullptr: count only
// (histogram of record byte hist_byte over the in-range items, e.g. the leading byte itself for the planner).
// Otherwise the in-range records are appended at records[*cursor ...) with one warp-aggregated atomic per 32 items
// (their order is irrelevant: equal keys are equal records up to the multiplicity bits, of which the emit takes the
// minimum).  Items beyond `capacity` are counted by the cursor but not stored.
template <int W>
__global__ void __launch_bounds__(256)
    k_s2s_extract_range(SeqsView sv, u32 k, u32 *__restrict__ records, u64 n_items, u32 lo, u32 hi,
                        unsigned long long *cursor, u64 capacity, u64 *hist, int hist_byte) {
  __shared__ u32 s_hist[256];
  for (int i = threadIdx.x; i < 256; i += 256) s_hist[i] = 0;
  __syncthreads();
  const u32 lane = threadIdx.x & 31;
  const u32 lt = lanemask_lt();
  for (u64 t0 = (u64)blockIdx.x * 256 + (threadIdx.x & ~31u); t0 < n_items; t0 += (u64)gridDim.x * 256) {  // warp-uniform
    const u64 t = t0 + lane;
    bool in = false;
    u32 rec[W];
    if (t < n_items) {
      u64 seq, rem;
      u32 L;
      const u32 *s;
      u32 nwords;
      if (sv.fixed_len) {
        L = sv.fixed_len;
        const u64 ips = 2ull * (L - k + 2);
        seq = t / ips;
        rem = t - seq * ips;
        nwords = div_ceil(L, 16);
        s = sv.words + seq * (sv.fixed_stride ? sv.fixed_stride : nwords);
      } else {
        u64 a = 0, b = sv.n_seqs;  // last seq with item_off[seq] <= t
        while (b - a > 1) {
          const u64 mid = (a + b) >> 1;
          if (sv.item_off[mid] <= t) a = mid; else b = mid;
        }
        seq = a;
        rem = t - sv.item_off[seq];
        L = sv.len[seq];
        nwords = div_ceil(L, 16);
        s = sv.words + sv.word_off[seq];
      }
      const u32 per_strand = L - k + 2;
      const u32 strand = rem >= per_strand ? 1u : 0u;
      const u32 offset = (u32)(rem - (u64)strand * per_strand);
      const u32 mult = sv.mult ? (u32)sv.mult[seq] : (s[sv.fixed_stride - 1] & 0xFFFFu);
      make_s2s_record<W>(s, nwords, L, k, strand, offset, mult, rec);
      const u32 top = rec[0] >> 16;  // the 8-base bucket id
      in = top >= lo && top <= hi;
    }
    const u32 mask = __ballot_sync(0xffffffffu, in);
    if (mask == 0) continue;
    if (records) {
      unsigned long long base = 0;
      if (lane == 0) base = atomicAdd(cursor, (unsigned long long)__popc(mask));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (in) {
        const u64 pos = base + __popc(mask & lt);
        if (pos < capacity) st_rec<W>(records, pos, rec);
      }
    }
    if (in && hist) atomicAdd(&s_hist[rec_byte<W>(rec, hist_byte)], 1u);
  }
  __syncthreads();
  if (hist)
    for (int i = threadIdx.x; i < 256; i += 256)
      if (s_hist[i]) atomicAdd((unsigned long long *)&hist[i], (unsigned long long)s_hist[i]);
}

// S-extract fast path: the sequences are `.edges` records of (k+1)-mers with k+1 <= 32 (the k_min case).  One
// thread turns one edge into its six sort items (both strands x offsets 0,1,2) with 64-bit arithmetic; strand 1
// is strand 0 of the reverse complement (seq_to_sdbg.cpp:672-690).  Item order matches k_s2s_extract.
template <int W>
__global__ void __launch_bounds__(256)
    k_s2s_extract_edges(const u32 *__restrict__ edges, u64 n_edges, u32 we, u32 k, u32 *__restrict__ records, u64 *hist,
                        int hist_byte) {
  __shared__ u32 s_hist[256];
  __shared__ __align__(16) u32 s_out[256 * 6 * W];  // the CTA's 1536 items, written out with coalesced 16 B stores
  for (int i = threadIdx.x; i < 256; i += 256) s_hist[i] = 0;
  __syncthreads();
  const u32 K1 = k + 1, T = 64u - 2u * K1;
  for (u64 base = (u64)blockIdx.x * 256; base < n_edges; base += (u64)gridDim.x * 256) {
    const u64 e = base + threadIdx.x;
    if (e < n_edges) {
      const u32 *ep = edges + e * we;
      const u32 e1 = we > 1 ? ep[1] : 0u;
      const u64 X0 = ((((u64)ep[0] << 32) | e1) >> T) << T;
      const u32 mult = ep[we - 1] & 0xFFFFu;
      const u64 R = ((u64)rev2((u32)X0) << 32) | rev2((u32)(X0 >> 32));  // reversed, right-aligned
      const u64 X1 = ((~R) << T);                                           // reverse complement, left-aligned
#pragma unroll
      for (int strand = 0; strand < 2; ++strand) {
        const u64 X = strand ? X1 : X0;
#pragma unroll
        for (int off = 0; off < 3; ++off) {
          const u32 nc = off == 2 ? k - 1 : k;
          const u64 chars = ((X << (2 * off)) >> (64 - 2 * nc)) << (64 - 2 * nc);
          const u32 prev = off == 0 ? kSentinel : (u32)(X >> (64 - 2 * off)) & 3u;
          const u32 low = ((off == 2 ? 0u : 1u) << 19) | (prev << 16) | (65535u - (off == 1 ? mult : 0u));
          u32 rec[W];
          rec[0] = (u32)(chars >> 32);
          if constexpr (W >= 2) rec[1] = (u32)chars;
#pragma unroll
          for (int j = 2; j < W; ++j) rec[j] = 0u;
          rec[W - 1] |= low;
          u32 *dst = s_out + (threadIdx.x * 6 + strand * 3 + off) * W;
#pragma unroll
          for (int j = 0; j < W; ++j) dst[j] = rec[j];
          if (hist) atomicAdd(&s_hist[rec_byte<W>(rec, hist_byte)], 1u);
        }
      }
    }
    __syncthreads();
    const u64 left = n_edges - base;
    const u32 nw = (u32)(left < 256 ? left : 256) * 6 * W;  // words this CTA produced; base*6*W*4 is 16 B aligned
    uint4 *gdst = reinterpret_cast<uint4 *>(records + base * 6 * W);
    const uint4 *ssrc = reinterpret_cast<const uint4 *>(s_out);
    for (u32 x = threadIdx.x; x < nw / 4; x += 256) gdst[x] = ssrc[x];
    for (u32 x = (nw & ~3u) + threadIdx.x; x < nw; x += 256) records[base * 6 * W + x] = s_out[x];
    __syncthreads();
  }
  if (hist)
    for (int i = threadIdx.x; i < 256; i += 256)
      if (s_hist[i]) atomicAdd((unsigned long long *)&hist[i], (unsigned long long)s_hist[i]);
}

// S-extract from `.edges` records WITH the in/out flags the count stage computed for them (aux bit0 = no solid
// incoming (k+2)-mer, bit1 = no outgoing): the $-items the emitter is certain to discard are not generated at all.
// An edge E = x0..xk yields, per strand, the items at offsets 0 ($ x0..x_{k-1}: "nothing enters this node"), 1 (the
// edge itself) and 2 (x2..xk $: "nothing leaves").  The emitter drops an offset-0 item when some edge y x0..x_{k-1}
// exists and an offset-2 item when some edge x1..xk z exists (seq_to_sdbg.cpp:760-776).  has_in(E) means a (k+2)-mer
// y E occurs >= m times, and every such occurrence contains y x0..x_{k-1} - a solid edge, in the set - so the
// offset-0 item of strand 0 (and, by the same argument on the reverse complement, the offset-2 item of strand 1) is
// provably discarded; likewise has_out(E) for offset 2 of strand 0 and offset 0 of strand 1.  Items that are merely
// LIKELY to be discarded (flag says "no in" but another edge enters the node) are still generated and left to the
// emitter, so the output is bit-identical; a genome at 30x keeps 2.02 of 6 items per edge.  Edges without flags
// (index >= n_aux: the mercy edges appended behind the solid ones) keep all six.  Items are appended at
// records[*cursor ...) in no particular order (one warp-aggregated atomic per 32 edges).
template <int W>
__global__ void __launch_bounds__(256)
    k_s2s_extract_edges_pruned(const u32 *__restrict__ edges, const uint8_t *__restrict__ aux, u64 n_edges, u64 n_aux, u32 we,
                               u32 k, u32 *__restrict__ records, unsigned long long *cursor, u64 capacity, u64 *hist,
                               int hist_byte) {
  __shared__ u32 s_hist[256];
  for (int i = threadIdx.x; i < 256; i += 256) s_hist[i] = 0;
  __syncthreads();
  const u32 lane = threadIdx.x & 31;
  for (u64 e0 = (u64)blockIdx.x * 256 + (threadIdx.x & ~31u); e0 < n_edges; e0 += (u64)gridDim.x * 256) {  // warp-uniform
    const u64 e = e0 + lane;
    u32 keep = 0;  // bit strand*3 + offset
    if (e < n_edges) {
      const u32 a = e < n_aux ? (u32)aux[e] : 3u;
      const u32 no_in = a & 1u, no_out = (a >> 1) & 1u;
      keep = (1u << 1) | (1u << 4) | (no_in << 0) | (no_out << 2) | (no_out << 3) | (no_in << 5);
    }
    const u32 cnt = (u32)__popc(keep);
    u32 inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 v = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= (u32)d) inc += v;
    }
    const u32 warp_total = __shfl_sync(0xffffffffu, inc, 31);
    unsigned long long base = 0;
    if (lane == 31) base = atomicAdd(cursor, (unsigned long long)warp_total);
    base = __shfl_sync(0xffffffffu, base, 31);
    if (cnt) {
      const u32 *ep = edges + e * we;
      const u32 mult = ep[we - 1] & 0xFFFFu;
      u64 dst = base + inc - cnt;
#pragma unroll
      for (u32 q = 0; q < 6; ++q) {
        if (!((keep >> q) & 1u)) continue;
        u32 rec[W];
        make_s2s_record<W>(ep, we, k + 1, k, q / 3, q % 3, mult, rec);
        if (dst < capacity) st_rec<W>(records, dst, rec);
        ++dst;
        if (hist) atomicAdd(&s_hist[rec_byte<W>(rec, hist_byte)], 1u);
      }
    }
  }
  __syncthreads();
  if (hist)
    for (int i = threadIdx.x; i < 256; i += 256)
      if (s_hist[i]) atomicAdd((unsigned long long *)&hist[i], (unsigned long long)s_hist[i]);
}

// ---- record field access (seq_to_sdbg.cpp:71-97) ----
template <int W>
__device__ __forceinline__ u32 s2s_a(const u32 (&r)[W], u32 k) {
  if ((r[W - 1] >> 19) & 1u) return (pick<W>(r, (k - 1) >> 4) >> (30 - 2 * ((k - 1) & 15))) & 3u;
  return kSentinel;
}
template <int W>
__device__ __forceinline__ u32 s2s_b(const u32 (&r)[W]) { return (r[W - 1] >> 16) & 7u; }

// IsDiffKMinusOneMer (seq_to_sdbg.cpp:46-69)
template <int W>
__device__ __forceinline__ bool diff_km1(const u32 (&x)[W], const u32 (&y)[W], u32 k) {
  const u32 bits = 2 * (k - 1);
  bool diff = false;
#pragma unroll
  for (int j = 0; j < W; ++j) {
    const int keep = (int)bits - 32 * j;
    const u32 m = keep <= 0 ? 0u : top_mask(keep > 32 ? 32u : (u32)keep);
    diff = diff || ((x[j] & m) != (y[j] & m));
  }
  return diff;
}

// Tip-label word q of a read2sdbg item (label_fmt = 1).  The items travel in the seq2sdbg layout (flags in the low 20
// bits of word W-1); the reference's stage-2 record (read_to_sdbg_s2.cpp:483-485, W1 = ceil((2k+4)/32) words) keeps
// nondollar<<3 | prev in the low 4 bits of word W1-1, and its tip label is the first ceil(k/16) raw words of THAT
// record (:602-606).  A tip has nondollar = 0, so the 4 flag bits are b.
__device__ __forceinline__ u32 r2s_label_word(u32 lw, u32 q, u32 W, u32 k, u32 b) {
  if (q == W - 1) lw &= 0xFFF00000u;
  if (q == div_ceil(2 * k + 4, 32) - 1) lw |= b;
  return lw;
}

struct EmitAcc {
  u32 bytes, items, tips, large;
};

// bucket_start holds the prefixes at each non-empty bucket's first item (~0 = empty); turn it into
// {byte offset, #items, #tips, #large} per bucket using the grand totals for the last bucket.  A bucket's extent ends
// where the NEXT NON-EMPTY bucket starts.  ONE block of 1024 threads, 64 consecutive buckets per thread: every thread
// finds the first non-empty bucket of its range, a suffix pass over the 1024 ranges gives the first non-empty bucket
// behind each range, then the thread walks its range backwards.  (The first version let every bucket scan forward for
// its successor: fine while all buckets are populated, but a rank of a multi-GPU build owns one contiguous range, and
// its last bucket then walked tens of thousands of empty buckets in one thread - 6 ms at 2 GPUs, 11 ms at 8.)
__global__ void __launch_bounds__(1024) k_bucket_finalize(const u64 *bucket_start, const u64 *totals, u64 *bucket_table) {
  constexpr u32 PER = MHB_NUM_BUCKETS / 1024;
  __shared__ u32 s_first[1024];
  const u32 t = threadIdx.x, b0 = t * PER;
  u32 first = 0xFFFFFFFFu;
  for (u32 i = 0; i < PER; ++i)
    if (first == 0xFFFFFFFFu && bucket_start[4ull * (b0 + i)] != ~0ull) first = b0 + i;
  s_first[t] = first;
  __syncthreads();
  if (t == 0) {  // s_first[r] := first non-empty bucket at or behind range r
    u32 run = 0xFFFFFFFFu;
    for (int r = 1023; r >= 0; --r) {
      if (s_first[r] != 0xFFFFFFFFu) run = s_first[r];
      s_first[r] = run;
    }
  }
  __syncthreads();
  u32 next = t + 1 < 1024 ? s_first[t + 1] : 0xFFFFFFFFu;  // first non-empty bucket behind my range
  for (int i = (int)PER - 1; i >= 0; --i) {
    const u32 b = b0 + (u32)i;
    const u64 *s = bucket_start + 4ull * b;
    u64 *o = bucket_table + 4ull * b;
    if (s[0] == ~0ull) {
      o[0] = o[1] = o[2] = o[3] = 0;
      continue;
    }
    u64 end[4];
    for (int q = 0; q < 4; ++q) end[q] = next != 0xFFFFFFFFu ? bucket_start[4ull * next + q] : totals[q];
    o[0] = s[0];
    o[1] = end[1] - s[1];
    o[2] = end[2] - s[2];
    o[3] = end[3] - s[3];
    next = b;
  }
}


// ------------------------------------------------------------------------------------------------
// S-emit v2 (A10): shared-memory staged, lane-blocked, no serial chain.
//
// A warp stages a chunk of 32*IPL sorted records (+ one record before, + a halo after) in shared memory with
// coalesced loads; lane l owns the (k-1)-mer groups whose first record lies in its IPL records and walks them
// out of shared memory (records beyond the halo come from global memory, so arbitrarily long groups stay
// correct).  Two walks: sizes -> warp scan -> items written to the chunk's compact slot of a scratch stream.
// Chunk totals are scanned (3-phase) and k_s2s_gather copies every chunk's bytes to its final offset.
// ------------------------------------------------------------------------------------------------
static constexpr int kEmit2Warps = 8, kEmit2Halo = 32;
__host__ __device__ constexpr int emit2_ipl(int w) { return w <= 4 ? 8 : (w <= 8 ? 4 : 2); }
__host__ __device__ constexpr int emit2_chunk(int w) { return 32 * emit2_ipl(w); }
__host__ __device__ constexpr int emit2_slots(int w) {  // staged record slots incl. one pad slot per IPL records
  return (1 + emit2_chunk(w) + kEmit2Halo) + (1 + emit2_chunk(w) + kEmit2Halo) / emit2_ipl(w) + 1;
}
__host__ __device__ inline u32 emit2_max_item_bytes(u32 k) { return 4u + 4u * words_per_tip_label(k); }

template <int W>
struct StagedRecs {
  const u32 *smem;  // staged window
  const u32 *glob;  // all records
  u64 a0;           // global index of staged slot 0
  u32 ns;           // staged records
  __device__ __forceinline__ void get(u64 t, u32 (&r)[W]) const {
    const u64 slot = t - a0;
    if (slot < ns) {
      const u32 *p = smem + ((u32)slot + (u32)slot / emit2_ipl(W)) * W;
#pragma unroll
      for (int j = 0; j < W; ++j) r[j] = p[j];
    } else {
      ld_rec<W>(glob, t, r);
    }
  }
};

// One thread walks the (k-1)-mer group that starts at record i (seq_to_sdbg.cpp:702-789) and either sizes (WRITE=false)
// or writes (WRITE=true: item bytes appended at out + acc.bytes) its SdBG items (sdbg_writer.cpp:25-58); returns the
// group's end.
template <int W, bool WRITE>
__device__ __forceinline__ u64 s2s_group2(const StagedRecs<W> &sr, u64 n, u64 i, u32 k, EmitAcc &acc, uint8_t *out,
                                          u32 *w_count, u32 &ones, u32 fmt) {
  const u32 WPT = words_per_tip_label(k);
  u32 r0[W], x[W];
  sr.get(i, r0);
  u32 hsa = 0, hsb = 0;
  u64 e = i;
  for (u64 j = i; j < n; ++j) {  // :724-738
    sr.get(j, x);
    if (j > i && diff_km1<W>(r0, x, k)) break;
    const u32 a = s2s_a<W>(x, k), b = s2s_b<W>(x);
    if (a != kSentinel && b != kSentinel) {
      hsa |= 1u << a;
      hsb |= 1u << b;
    }
    e = j + 1;
  }
  u32 outputed_b = 0;
  u64 j = i;
  u32 cur[W];
#pragma unroll
  for (int q = 0; q < W; ++q) cur[q] = r0[q];
  while (j < e) {  // :740-786
    const u32 a = s2s_a<W>(cur, k), b = s2s_b<W>(cur);
    u64 t = j + 1;
    u32 na = 0xFF, nb = 0xFF;
    u32 nx[W];
    u32 best = cur[W - 1] & 0xFFFFu;
    while (t < e) {
      sr.get(t, nx);
      na = s2s_a<W>(nx, k);
      nb = s2s_b<W>(nx);
      if (na != a || nb != b) break;
      best = min(best, nx[W - 1] & 0xFFFFu);
      ++t;
    }
    const bool more = t < e;
    const bool skip = (a == kSentinel && ((hsb >> b) & 1u)) || (b == kSentinel && ((hsa >> a) & 1u));
    if (!skip) {
      const u32 w = (b == kSentinel) ? 0u : (((outputed_b >> b) & 1u) ? b + 5u : b + 1u);
      u32 last = 0;
      if (a != kSentinel) last = (b == kSentinel) ? 1u : ((!more || na != a || nb == kSentinel) ? 1u : 0u);
      outputed_b |= 1u << b;
      const u32 mul = 65535u - best;
      const u32 tip = a == kSentinel ? 1u : 0u;
      const u32 sz = 2u + (mul > 254u ? 2u : 0u) + (tip ? 4u * WPT : 0u);
      if (WRITE) {
        uint16_t *o = reinterpret_cast<uint16_t *>(out + acc.bytes);
        o[0] = (uint16_t)((w | (last << 4) | (tip << 5)) | ((mul > 255u ? 255u : mul) << 8));
        u32 p = 1;
        if (mul > 254u) o[p++] = (uint16_t)mul;
        if (tip) {
          for (u32 q = 0; q < WPT; ++q) {
            u32 lw = pick<W>(cur, q);
            if (fmt) lw = r2s_label_word(lw, q, (u32)W, k, b);
            else if (q == (u32)W - 1) lw = (lw & 0xFFFF0000u) | best;  // label = raw words of the run's first sorted record
            o[p++] = (uint16_t)(lw & 0xFFFFu);
            o[p++] = (uint16_t)(lw >> 16);
          }
        }
        atomicAdd(&w_count[w], 1u);
        ones += last;
      }
      acc.bytes += sz;
      acc.items += 1;
      acc.tips += tip;
      acc.large += mul > 254u ? 1u : 0u;
    }
    j = t;
    if (more) {
#pragma unroll
      for (int q = 0; q < W; ++q) cur[q] = nx[q];
    }
  }
  return e;
}

template <int W>
__global__ void __launch_bounds__(kEmit2Warps * 32)
    k_s2s_judge(const u32 *__restrict__ recs, u64 n, u32 k, u32 n_chunks, uint8_t *__restrict__ tmp,
                u32 *__restrict__ chunk_tot /*4 planes of n_chunks*/, u32 *__restrict__ bucket_local /*65536 x 5*/,
                u64 *totals, u32 fmt) {
  constexpr int IPL = emit2_ipl(W), CH = emit2_chunk(W);
  extern __shared__ __align__(16) u32 smem_e[];
  __shared__ u32 s_w[9];
  const u32 lane = lane_id(), warp = threadIdx.x >> 5;
  u32 *my = smem_e + (size_t)warp * emit2_slots(W) * W;
  if (threadIdx.x < 9) s_w[threadIdx.x] = 0;
  __syncthreads();
  const u32 maxb = emit2_max_item_bytes(k);
  u32 ones = 0;
  for (u64 chunk = (u64)blockIdx.x * kEmit2Warps + warp; chunk < n_chunks; chunk += (u64)gridDim.x * kEmit2Warps) {
    const u64 a = chunk * CH;
    const u64 b = a + CH < n ? a + CH : n;
    const u64 a0 = a > 0 ? a - 1 : 0;
    const u64 hi = a + CH + kEmit2Halo < n ? a + CH + kEmit2Halo : n;
    const u32 ns = (u32)(hi - a0);
    __syncwarp();
    for (u32 t = lane; t < ns; t += 32) {
      u32 r[W];
      ld_rec<W>(recs, a0 + t, r);
      u32 *dst = my + (t + t / IPL) * W;
#pragma unroll
      for (int j = 0; j < W; ++j) dst[j] = r[j];
    }
    __syncwarp();
    const StagedRecs<W> sr{my, recs, a0, ns};

    // this lane's first group head (if any) in [lo, hi_l)
    const u64 lo = a + (u64)lane * IPL;
    const u64 hi_l = lo + IPL < b ? lo + IPL : b;
    u64 first = hi_l;
    if (lo < b) {
      u32 p[W], c[W];
      if (lo > 0) sr.get(lo - 1, p);
      for (u64 t = lo; t < hi_l; ++t) {
        sr.get(t, c);
        if (t == 0 || diff_km1<W>(p, c, k)) {
          first = t;
          break;
        }
#pragma unroll
        for (int q = 0; q < W; ++q) p[q] = c[q];
      }
    }
    // walk 1: sizes
    EmitAcc acc = {0, 0, 0, 0};
    u32 dummy = 0;
    for (u64 t = first; t < hi_l;) t = s2s_group2<W, false>(sr, n, t, k, acc, nullptr, nullptr, dummy, fmt);
    // lane prefixes + chunk totals
    u32 inc[4] = {acc.bytes, acc.items, acc.tips, acc.large};
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const u32 v = __shfl_up_sync(0xffffffffu, inc[q], d);
        if (lane >= (u32)d) inc[q] += v;
      }
    }
    if (lane == 31) {
#pragma unroll
      for (int q = 0; q < 4; ++q) chunk_tot[(u64)q * n_chunks + chunk] = inc[q];
    }
    const u32 pre[4] = {inc[0] - acc.bytes, inc[1] - acc.items, inc[2] - acc.tips, inc[3] - acc.large};
    // walk 2: write items into the chunk's compact slot; note where each bucket starts
    uint8_t *out = tmp + chunk * (u64)CH * maxb + pre[0];
    EmitAcc wacc = {0, 0, 0, 0};
    for (u64 t = first; t < hi_l;) {
      u32 h[W], pv[W];
      sr.get(t, h);
      const u32 bucket = h[0] >> 16;
      bool new_bucket = t == 0;
      if (t > 0) {
        sr.get(t - 1, pv);
        new_bucket = (pv[0] >> 16) != bucket;
      }
      if (new_bucket) {
        u32 *bl = bucket_local + 5ull * bucket;
        bl[0] = (u32)chunk;
        bl[1] = pre[0] + wacc.bytes;
        bl[2] = pre[1] + wacc.items;
        bl[3] = pre[2] + wacc.tips;
        bl[4] = pre[3] + wacc.large;
      }
      t = s2s_group2<W, true>(sr, n, t, k, wacc, out, s_w, ones, fmt);
    }
  }
  for (int d = 16; d; d >>= 1) ones += __shfl_xor_sync(0xffffffffu, ones, d);
  if (lane == 0 && ones) atomicAdd((unsigned long long *)&totals[13], (unsigned long long)ones);
  __syncthreads();
  if (threadIdx.x < 9 && s_w[threadIdx.x])
    atomicAdd((unsigned long long *)&totals[4 + threadIdx.x], (unsigned long long)s_w[threadIdx.x]);
}

// copy every chunk's compact bytes to their final position (all sizes and offsets are even)
__global__ void __launch_bounds__(256)
    k_s2s_gather(const uint8_t *__restrict__ tmp, u32 chunk_records, u32 maxb, u32 n_chunks,
                 const u32 *__restrict__ chunk_bytes, const u64 *__restrict__ chunk_off, uint8_t *__restrict__ out,
                 u64 capacity) {
  const u32 lane = lane_id();
  for (u64 chunk = (u64)blockIdx.x * 8 + (threadIdx.x >> 5); chunk < n_chunks; chunk += (u64)gridDim.x * 8) {
    const u32 nb = chunk_bytes[chunk];
    const u64 off = chunk_off[chunk];
    if (off + nb > capacity) continue;
    const uint16_t *src = reinterpret_cast<const uint16_t *>(tmp + chunk * (u64)chunk_records * maxb);
    uint16_t *dst = reinterpret_cast<uint16_t *>(out + off);
    for (u32 x = lane; x < nb / 2; x += 32) dst[x] = src[x];
  }
}

// bucket_local {chunk, bytes, items, tips, large within the chunk} + the chunks' global offsets -> bucket_start
__global__ void k_bucket_starts(const u32 *bucket_local, const u64 *chunk_off /*4 planes*/, u64 n_chunks, u64 *bucket_start) {
  for (u32 b = blockIdx.x * blockDim.x + threadIdx.x; b < MHB_NUM_BUCKETS; b += gridDim.x * blockDim.x) {
    const u32 *bl = bucket_local + 5ull * b;
    u64 *o = bucket_start + 4ull * b;
    if (bl[0] == 0xFFFFFFFFu) {
      o[0] = o[1] = o[2] = o[3] = ~0ull;
    } else {
      for (int q = 0; q < 4; ++q) o[q] = chunk_off[(u64)q * n_chunks + bl[0]] + bl[1 + q];
    }
  }
}

}  // namespace mhb
