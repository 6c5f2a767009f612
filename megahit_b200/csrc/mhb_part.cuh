// mhb_part.cuh -- UNSTABLE radix partition pass: the first pass of an LSD sort (and any stand-alone partition) has no
// earlier order to preserve, so it needs neither the decoupled look-back chain nor stable ranking.
//   * a tile's place inside every digit's output region is reserved with one global atomicAdd per digit (256 per tile,
//     all in flight together) - tiles never wait for each other;
//   * a record's rank inside its tile comes from one shared-memory atomic (no eight-ballot peer search, no per-warp
//     counter rows, no warp-base pass);
//   * reorder in shared memory + coalesced scatter + the next pass's digit histogram as in k_radix_pass3.
// Which of several equal-digit records lands first depends on scheduling; callers that need a deterministic total
// order of FULLY equal sort keys must use the stable pass (the public mhb_sort_records does).  The count and seq2sdbg
// stages do not: records with equal sort keys are tallied (kmer_counter.cpp:279-305) or reduced to their minimum
// multiplicity (seq_to_sdbg.cpp:760-785) whatever their order.
#pragma once
#include "mhb_sort3.cuh"

namespace mhb {

__device__ __forceinline__ u32 atom_shared_inc_ret(u32 *p) {
  u32 old;
  asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(p)) : "memory");
  return old;
}

template <int WR>
struct PartCfg {
  static constexpr int THREADS = 384;
  static constexpr int IPT = SortCfg3<WR>::IPT;
  static constexpr int TILE = THREADS * IPT;
  static constexpr size_t SMEM = 256 * 8 /*s_base*/ + 4 * 256 * 4 /*s_cnt, s_off, s_cur, s_next*/ + 16 * 4 + (size_t)TILE * WR * 4;
  static constexpr size_t SMEM_OWNER_HIST = SMEM + 16 * 256 * 4;  // + per-owner histograms of the next sort byte
};

// OWNER_LUT + HAS_NEXT: the digit is the owning rank (<= 16) and next_hist is [16][256]: one histogram of record byte
// `next_byte` PER OWNER, so that the receiving rank gets the first-pass histogram of its sort for free.
template <int WR, bool OWNER_LUT, bool HAS_NEXT>
__global__ void __launch_bounds__(PartCfg<WR>::THREADS, 2)
    k_part_unstable(const u32 *__restrict__ in, u64 n, u32 num_tiles, int byte_idx,
                    const u64 *__restrict__ bin_addr /*byte address of each digit's first output record*/,
                    unsigned long long *gcursor /*[256], zeroed: records of each digit placed so far*/, u32 *tile_counter,
                    u64 *next_hist, int next_byte, const uint8_t *__restrict__ digit_lut) {
  constexpr bool OWNER_HIST = OWNER_LUT && HAS_NEXT;
  using C = PartCfg<WR>;
  constexpr int THREADS = C::THREADS, IPT = C::IPT, TILE = C::TILE;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  u64 *s_base = reinterpret_cast<u64 *>(smem_raw);  // 256: byte address of this tile's slot inside digit d's region
  u32 *s_cnt = reinterpret_cast<u32 *>(s_base + 256);
  u32 *s_off = s_cnt + 256;   // exclusive scan of s_cnt: the digit's first position inside the reordered tile
  u32 *s_cur = s_off + 256;   // running cursor while ranking
  u32 *s_next = s_cur + 256;
  u32 *s_misc = s_next + 256;  // 16
  u32 *s_recs = s_misc + 16;
  u32 *s_onext = s_recs + (size_t)C::TILE * WR;  // OWNER_HIST: [16][256]
  __shared__ uint8_t s_lut[OWNER_LUT ? 256 : 1];
  const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u32 widx = (u32)(WR - 1 - (byte_idx >> 2)), bsel = (u32)(byte_idx & 3);
  const u32 nwidx = (u32)(WR - 1 - (next_byte >> 2)), nbsel = (u32)(next_byte & 3);
  for (int i = tid; i < 256; i += THREADS) {
    s_cnt[i] = 0;
    s_next[i] = 0;
  }
  if constexpr (OWNER_HIST) {
    for (int i = tid; i < 16 * 256; i += THREADS) s_onext[i] = 0;
  }
  if constexpr (OWNER_LUT) {
    for (int i = tid; i < 256; i += THREADS) s_lut[i] = digit_lut[i];
  }
  if (tid == 0) s_misc[0] = atomicAdd(tile_counter, 1u);
  __syncthreads();
  u32 tile = s_misc[0];
  while (tile < num_tiles) {
    u32 next_ticket = 0;
    if (tid == 0) next_ticket = atomicAdd(tile_counter, 1u);
    const u64 tile_base = (u64)tile * TILE;
    const u32 valid = tile_base + TILE <= n ? (u32)TILE : (u32)(n - tile_base);
    // ---- load (warp-striped) + tile histogram ----
    u32 r[IPT][WR];
    u32 dg[IPT];
    const u32 wbase = warp * 32 * IPT + lane;
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
      const u32 p = wbase + (u32)i * 32;
      if (p < valid) ld_rec_pinned<WR>(in, tile_base + p, r[i]);
    }
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
      const u32 p = wbase + (u32)i * 32;
      u32 d = 0;
      if (p < valid) {
        d = rec_digit<WR>(r[i], widx, bsel);
        if constexpr (OWNER_LUT) d = s_lut[d];
        red_shared_inc(&s_cnt[d]);
      }
      dg[i] = d;
    }
    __syncthreads();
    // ---- reserve the tile's slot in every digit's region; positions inside the tile ----
    if (tid < 256) {
      const u32 c = s_cnt[tid];
      const unsigned long long g = c ? atomicAdd(&gcursor[tid], (unsigned long long)c) : 0ull;
      u32 inc = c;
#pragma unroll
      for (int dd = 1; dd < 32; dd <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, inc, dd);
        if (lane >= (u32)dd) inc += t;
      }
      if (lane == 31) s_misc[4 + warp] = inc;
      s_off[tid] = inc - c;  // completed below
      s_base[tid] = bin_addr[tid] + g * (u64)(WR * 4);
    }
    __syncthreads();
    if (tid < 256) {
      u32 add = 0;
#pragma unroll
      for (int w = 0; w < 7; ++w) add += (warp > (u32)w) ? s_misc[4 + w] : 0u;
      const u32 o = s_off[tid] + add;
      s_off[tid] = o;
      s_cur[tid] = o;
    }
    if (tid == 0) s_misc[0] = next_ticket;
    __syncthreads();
    // ---- rank (one shared-memory atomic per record) + reorder ----
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
      const u32 p = wbase + (u32)i * 32;
      if (p < valid) st_shared_rec<WR>(s_recs, atom_shared_inc_ret(&s_cur[dg[i]]), r[i]);
    }
    __syncthreads();
    const u32 next_tile = s_misc[0];
    // ---- coalesced scatter + next digit's histogram ----
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
      const u32 p = (u32)i * THREADS + tid;
      if (p < valid) {
        u32 q[WR];
        ld_rec<WR>(s_recs, p, q);
        u32 dd = rec_digit<WR>(q, widx, bsel);
        if constexpr (OWNER_LUT) dd = s_lut[dd];
        st_global_rec<WR>(s_base[dd] + (u64)(p - s_off[dd]) * (WR * 4), q);
        if constexpr (OWNER_HIST) red_shared_inc(&s_onext[(dd & 15u) * 256 + rec_digit<WR>(q, nwidx, nbsel)]);
        else if constexpr (HAS_NEXT) red_shared_inc(&s_next[rec_digit<WR>(q, nwidx, nbsel)]);
      }
    }
    for (int i = tid; i < 256; i += THREADS) s_cnt[i] = 0;
    __syncthreads();
    tile = next_tile;
  }
  if constexpr (OWNER_HIST) {
    for (int i = tid; i < 16 * 256; i += THREADS)
      if (s_onext[i]) atomicAdd((unsigned long long *)&next_hist[i], (unsigned long long)s_onext[i]);
  } else if constexpr (HAS_NEXT) {
    for (int i = tid; i < 256; i += THREADS)
      if (s_next[i]) atomicAdd((unsigned long long *)&next_hist[i], (unsigned long long)s_next[i]);
  }
}

}  // namespace mhb
