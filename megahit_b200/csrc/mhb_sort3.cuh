// mhb_sort3.cuh -- the stable radix pass.  One pass = one persistent kernel: every CTA repeatedly claims the next tile
// (atomic ticket, so tiles start in order), ranks its records by digit with warp ballots and per-warp shared-memory
// counters, publishes the tile's per-digit counts and resolves its global offsets by decoupled look-back over earlier
// tiles, reorders the tile in shared memory so that every digit's records are contiguous, and scatters them with
// coalesced stores.  While the records are in registers the pass also accumulates the histogram of the NEXT pass's
// digit, so the input is never read just to count.
//
// The round-1 pass was issue-bound at ~125 thread-instructions per record (profiles/r1_radix_v2_*.txt: 24 %
// issue-active with 2 CTAs/SM, DRAM traffic 1.01x algorithmic), of which only ~26 were the eight ballots.  This one
// removes what surrounded them:
//   * the next tile's ticket is requested a whole tile ahead (the global atomic's latency is never exposed);
//   * per-warp digit counters are read by ALL lanes before the leader bumps them (no shuffle, no divergent load);
//   * the prefix over warps, the tile scan and the fold of the digit's start run as ONE pass of 256 threads
//     (6 block barriers per tile instead of 9, no separate fold loop, no s_bin_start array);
//   * a tile's digit counts are histogrammed and published right after its load, before ranking (early publish);
//   * full tiles take a scatter path without per-record bounds checks;
//   * counters are cleared with 128-bit stores while the scatter's global stores are in flight.
// Measured on B200, 1.23 G 8-byte records, this pass takes 6.44 ms; other tile shapes, shared-memory OR-match ranking,
// register prefetch of the next tile, batched shared-memory loads, wider or narrower look-back windows, compact
// look-back descriptors and two-stream ranking were all slower (profiles/r1d_sort_sweep.txt, profiles/r2a_sort_sweep.json).
#pragma once
#include "mhb_sort.cuh"

namespace mhb {

// Tile geometry: 384 threads, 2 CTAs/SM, records per thread by width so that a tile's records fill ~55 KB of shared memory
template <int WR>
struct SortCfg3 {
  static constexpr int THREADS = 384;
  static constexpr int MIN_BLOCKS = 2;
  static constexpr int IPT = WR <= 2 ? 18 : (WR <= 3 ? 12 : (WR <= 4 ? 10 : (WR <= 6 ? 6 : (WR <= 9 ? 4 : 2))));
  static constexpr int TILE = THREADS * IPT;
  static constexpr int NW = THREADS / 32;
  static constexpr int LBW = 2;  // look-back descriptors fetched per round trip; the first window is fetched before the reorder
  static constexpr size_t SMEM = 256 * 8 /*s_glob*/ + (size_t)NW * 256 * 4 /*counters*/ + 256 * 4 /*s_next*/ +
                                 256 * 4 /*s_early*/ + 16 * 4 /*misc*/ + (size_t)TILE * WR * 4;
};

// a tile's record loads, issued where they stand: asm volatile keeps the compiler from moving them past the shared-memory
// work around them
template <int WR>
__device__ __forceinline__ void ld_rec_pinned(const u32 *base, u64 idx, u32 (&r)[WR]) {
  const u32 *p = base + idx * WR;
  if constexpr (WR % 4 == 0) {
#pragma unroll
    for (int j = 0; j < WR; j += 4)
      asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];"
                   : "=r"(r[j]), "=r"(r[j + 1]), "=r"(r[j + 2]), "=r"(r[j + 3])
                   : "l"(p + j));
  } else if constexpr (WR % 2 == 0) {
#pragma unroll
    for (int j = 0; j < WR; j += 2) asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];" : "=r"(r[j]), "=r"(r[j + 1]) : "l"(p + j));
  } else {
#pragma unroll
    for (int j = 0; j < WR; ++j) asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(r[j]) : "l"(p + j));
  }
}

// Stores/reductions issued from the unrolled reorder / scatter loops of the partition pass (mhb_part.cuh).  As plain
// C++ they would be generic-address stores that may alias shared memory, which forces the compiler to serialise "load
// record i+1" behind "store record i"; as asm without a memory clobber the shared-memory loads of a whole chunk are issued back to back (the kernel is
// latency-bound at 2 CTAs/SM, so every exposed 30-cycle LDS round trip counts).  Nothing read inside those loops is
// written by them: the reordered records and the digit bases are complete before the barrier that precedes the scatter.
template <int WR>
__device__ __forceinline__ void st_global_rec(u64 addr, const u32 (&q)[WR]) {
  if constexpr (WR % 4 == 0) {
#pragma unroll
    for (int j = 0; j < WR; j += 4)
      asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(addr + 4 * j), "r"(q[j]), "r"(q[j + 1]), "r"(q[j + 2]), "r"(q[j + 3]));
  } else if constexpr (WR % 2 == 0) {
#pragma unroll
    for (int j = 0; j < WR; j += 2) asm volatile("st.global.v2.u32 [%0], {%1, %2};" ::"l"(addr + 4 * j), "r"(q[j]), "r"(q[j + 1]));
  } else {
#pragma unroll
    for (int j = 0; j < WR; ++j) asm volatile("st.global.u32 [%0], %1;" ::"l"(addr + 4 * j), "r"(q[j]));
  }
}
__device__ __forceinline__ void red_shared_inc(u32 *p) {
  asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(smem_u32(p)));
}
template <int WR>
__device__ __forceinline__ void st_shared_rec(u32 *base, u32 idx, const u32 (&q)[WR]) {
  const u32 a = smem_u32(base) + idx * (WR * 4);
  if constexpr (WR % 4 == 0) {
#pragma unroll
    for (int j = 0; j < WR; j += 4)
      asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a + 4 * j), "r"(q[j]), "r"(q[j + 1]), "r"(q[j + 2]), "r"(q[j + 3]));
  } else if constexpr (WR % 2 == 0) {
#pragma unroll
    for (int j = 0; j < WR; j += 2) asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a + 4 * j), "r"(q[j]), "r"(q[j + 1]));
  } else {
#pragma unroll
    for (int j = 0; j < WR; ++j) asm volatile("st.shared.u32 [%0], %1;" ::"r"(a + 4 * j), "r"(q[j]));
  }
}

// Optional per-tile timeline (diagnostic build only: `make timeline` -> libmhb_timeline.so, -DMHB_SORT_TIMELINE; the
// production library contains none of this).  One 16-word row per tile: tile, SM id, globaltimer at the tile's start,
// then clock64 deltas from the start at: records in registers, early publish done, ranking done (B1), warp bases
// done (B3), reorder done, look-back done, B4 passed, scatter done (B5); then max / sum over the 256 digit threads of
// the descriptors examined and of the re-polls of unpublished descriptors.
#ifdef MHB_SORT_TIMELINE
__device__ unsigned long long *g_sort_timeline = nullptr;
__device__ unsigned long long g_sort_timeline_rows = 0;
#define MHB_TL_DECL                                                                             \
  __shared__ unsigned int s_tl_depth_max, s_tl_depth_sum, s_tl_spin_max, s_tl_spin_sum;         \
  unsigned long long tl_t0 = 0, tl_g0 = 0, tl_v[8] = {0, 0, 0, 0, 0, 0, 0, 0};                  \
  unsigned int tl_depth = 0, tl_spin = 0;
#define MHB_TL_START()                                                                          \
  do {                                                                                          \
    if (tid == 0) {                                                                             \
      tl_t0 = clock64();                                                                        \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tl_g0));                                 \
      s_tl_depth_max = s_tl_depth_sum = s_tl_spin_max = s_tl_spin_sum = 0;                      \
    }                                                                                           \
    tl_depth = tl_spin = 0;                                                                     \
  } while (0)
#define MHB_TL_MARK(i)                         \
  do {                                         \
    if (tid == 0) tl_v[i] = clock64() - tl_t0; \
  } while (0)
#define MHB_TL_DEPTH() (++tl_depth)
#define MHB_TL_SPIN() (++tl_spin)
#define MHB_TL_LB_DONE()                       \
  do {                                         \
    atomicMax(&s_tl_depth_max, tl_depth);      \
    atomicAdd(&s_tl_depth_sum, tl_depth);      \
    atomicMax(&s_tl_spin_max, tl_spin);        \
    atomicAdd(&s_tl_spin_sum, tl_spin);        \
  } while (0)
#define MHB_TL_FLUSH()                                                                          \
  do {                                                                                          \
    if (tid == 0 && g_sort_timeline && (unsigned long long)tile < g_sort_timeline_rows) {       \
      unsigned long long *row = g_sort_timeline + (unsigned long long)tile * 16;                \
      unsigned int smid;                                                                        \
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));                                         \
      row[0] = tile;                                                                            \
      row[1] = smid;                                                                            \
      row[2] = tl_g0;                                                                           \
      for (int q_ = 0; q_ < 8; ++q_) row[3 + q_] = tl_v[q_];                                    \
      row[11] = s_tl_depth_max;                                                                 \
      row[12] = s_tl_depth_sum;                                                                 \
      row[13] = s_tl_spin_max;                                                                  \
      row[14] = s_tl_spin_sum;                                                                  \
      row[15] = blockIdx.x;                                                                     \
    }                                                                                           \
  } while (0)
#else
#define MHB_TL_DECL
#define MHB_TL_START() ((void)0)
#define MHB_TL_MARK(i) ((void)0)
#define MHB_TL_DEPTH() ((void)0)
#define MHB_TL_SPIN() ((void)0)
#define MHB_TL_LB_DONE() ((void)0)
#define MHB_TL_FLUSH() ((void)0)
#endif

template <int WR, bool HAS_NEXT = true>
__global__ void __launch_bounds__(SortCfg3<WR>::THREADS, SortCfg3<WR>::MIN_BLOCKS)
    k_radix_pass3(const u32 *__restrict__ in, u64 n, u32 num_tiles, int byte_idx,
                  const u64 *__restrict__ bin_addr /*byte address of each digit's first output record*/, u64 *lookback,
                  u32 *tile_counter, u64 *next_hist, int next_byte, u32 epoch) {
  using C = SortCfg3<WR>;
  constexpr int THREADS = C::THREADS, IPT = C::IPT, TILE = C::TILE, NW = C::NW, LBW = C::LBW;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  u64 *s_glob = reinterpret_cast<u64 *>(smem_raw);        // 256: byte address of the digit's slot for tile position 0
  u32 *s_cnt = reinterpret_cast<u32 *>(s_glob + 256);     // NW * 256
  u32 *s_next = s_cnt + NW * 256;                         // 256
  u32 *s_early = s_next + 256;                            // 256: tile digit counts taken right after the load
  u32 *s_misc = s_early + 256;                            // 16: [0] ticket, [4..12] scan
  u32 *s_recs = s_misc + 16;                              // TILE * WR (16-byte aligned)

  const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u32 lt_mask = lanemask_lt();
  const u32 widx = (u32)(WR - 1 - (byte_idx >> 2)), bsel = (u32)(byte_idx & 3);
  const u32 nwidx = (u32)(WR - 1 - (next_byte >> 2)), nbsel = (u32)(next_byte & 3);
  u32 *my_cnt = s_cnt + warp * 256;
  MHB_TL_DECL

  for (int i = tid; i < 256; i += THREADS) s_next[i] = 0;
  for (int i = tid; i < 256; i += THREADS) s_early[i] = 0;
  for (int i = tid; i < NW * 256; i += THREADS) s_cnt[i] = 0;
  if (tid == 0) s_misc[0] = atomicAdd(tile_counter, 1u);
  __syncthreads();
  u32 tile = s_misc[0];

  // ---- load (warp-striped: slot i of lane l = warp chunk[i*32 + l]) ----
  u32 r[IPT][WR];
  auto load_tile = [&](u32 t) {
    const u64 tb = (u64)t * TILE;
    const u64 warp_base = tb + (u64)warp * 32 * IPT + lane;
    if (tb + TILE <= n) {
#pragma unroll
      for (int i = 0; i < IPT; ++i) ld_rec_pinned<WR>(in, warp_base + (u64)i * 32, r[i]);
    } else {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const u64 idx = warp_base + (u64)i * 32;
        if (idx < n) {
          ld_rec_pinned<WR>(in, idx, r[i]);
        } else {
#pragma unroll
          for (int j = 0; j < WR; ++j) r[i][j] = 0xFFFFFFFFu;  // padding sorts to the very end of the tile
        }
      }
    }
  };

  while (tile < num_tiles) {
    // ticket of the NEXT tile: requested now, stored to shared memory just before this tile's last barrier, so the
    // global atomic's latency is never waited for.  Tickets are still handed out in start order (a CTA only ever
    // waits on smaller tickets than the ones it holds), so the look-back cannot deadlock.
    u32 next_ticket = 0;
    MHB_TL_START();
    if (tid == 0) next_ticket = atomicAdd(tile_counter, 1u);
    const u64 tile_base = (u64)tile * TILE;
    const bool full = tile_base + TILE <= n;
    const u32 valid = full ? (u32)TILE : (u32)(n - tile_base);

    load_tile(tile);

    // ---- early publish: histogram the tile's digits and publish the counts now, a whole rank phase before the tile
    // needs its predecessors: when the following tiles look back, this descriptor is already there (no spinning on
    // "invalid")
#ifdef MHB_SORT_TIMELINE
    if (tid == 0) {  // first use of the tile's records: the wait for the loads ends here
      volatile u32 sink = r[0][0];
      (void)sink;
      tl_v[0] = clock64() - tl_t0;
    }
#endif
#pragma unroll
    for (int i = 0; i < IPT; ++i) red_shared_inc(&s_early[rec_digit<WR>(r[i], widx, bsel)]);
    __syncthreads();
    if (tid < 256) {
      // padding records all carry digit 255 and are not real: exclude them from what we publish
      const u32 c = s_early[tid] - ((tid == 255) ? (u32)(TILE - valid) : 0u);
      st_relaxed(lookback + (u64)tile * 256 + tid, (tile == 0 ? kLbInclusive : kLbPartial) | lb_epoch(epoch) | (u64)c);
    }

    MHB_TL_MARK(1);
    // ---- rank inside the warp: rk = rank among the warp's records with the same digit << 8 | digit.  The lanes
    // holding the same digit come from eight ballots, one per digit bit: constant cost, no shared-memory traffic ----
    u32 rk[IPT];
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
      const u32 d = rec_digit<WR>(r[i], widx, bsel);
      u32 peers = 0xffffffffu;
#pragma unroll
      for (int bit = 0; bit < 8; ++bit) {
        u32 mask;
        asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\t"
            "vote.sync.ballot.b32 %0, p, 0xffffffff;\n\t@!p not.b32 %0, %0;\n\t}"
            : "=r"(mask)
            : "r"(d), "r"(1u << bit));
        peers &= mask;
      }
      volatile u32 *slot = my_cnt + d;
      const u32 old = *slot;  // every lane reads the running count before the leader bumps it
      __syncwarp();
      const u32 below = __popc(peers & lt_mask);
      if ((peers >> lane) <= 1u) *slot = old + below + 1u;  // highest peer lane: below + 1 = popc(peers)
      __syncwarp();
      rk[i] = ((old + below) << 8) | d;
    }
    __syncthreads();  // B1: all warps' counters final
    MHB_TL_MARK(2);

    // ---- per digit (threads 0..255): tile total, scan over digits, warp bases; first look-back window ----
    u32 total = 0, excl = 0;
    if (tid < 256) {
#pragma unroll
      for (int w = 0; w < NW; ++w) total += s_cnt[w * 256 + tid];
      u32 inc = total;
#pragma unroll
      for (int dd = 1; dd < 32; dd <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, inc, dd);
        if (lane >= (u32)dd) inc += t;
      }
      if (lane == 31) s_misc[4 + warp] = inc;
      excl = inc - total;
    }
    __syncthreads();  // B2
    u32 pub = 0;
    u64 win[LBW];
    if (tid == 0) s_misc[0] = next_ticket;  // requested a whole rank phase ago: no wait
    if (tid < 256) {
#pragma unroll
      for (int w = 0; w < 7; ++w) excl += (warp > (u32)w) ? s_misc[4 + w] : 0u;
      pub = total - ((tid == 255) ? (u32)(TILE - valid) : 0u);
#pragma unroll
      for (int j = 0; j < LBW; ++j)
        win[j] = (tile > (u32)j) ? ld_relaxed(lookback + (u64)(tile - 1 - j) * 256 + tid) : 0ull;
      // counters become: position in the tile of the warp's first record with this digit
      u32 run = excl;
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        const u32 c = s_cnt[w * 256 + tid];
        s_cnt[w * 256 + tid] = run;
        run += c;
      }
    }
    __syncthreads();  // B3
    MHB_TL_MARK(3);

    // ---- reorder in shared memory: every digit's records become contiguous, input order kept ----
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
      const u32 pos = my_cnt[rk[i] & 255u] + (rk[i] >> 8);
      st_rec<WR>(s_recs, pos, r[i]);
    }
    MHB_TL_MARK(4);
    const u32 next_tile = s_misc[0];  // written before B3, rewritten only after the next tile's B1

    // ---- global offsets by decoupled look-back.  All CTAs run the same phases almost in step, so the nearest
    // predecessors are still "partial" when a tile looks back and the walk to the last "inclusive" descriptor is long
    // (profiles/r1b: 25 % of all warp samples were this loop + the CTA waiting for it at B4).  The walk therefore
    // fetches LBW descriptors at a time - all loads in flight together, one round trip per LBW predecessors; the first
    // window was requested before the reorder.
    if (tid < 256) {
      u64 prefix = 0;
      if (tile > 0) {
        const u64 epv = lb_epoch(epoch);
        u32 p = tile - 1;  // descriptor win[0] belongs to tile p
        bool done = false;
#pragma unroll
        for (int j = 0; j < LBW; ++j) {
          if (!done) {
            u64 v = win[j];
            const u64 *pp = lookback + (u64)(p - j) * 256 + tid;
            MHB_TL_DEPTH();
            while ((v & kLbStatusMask) == 0 || (v & lb_epoch(255)) != epv) {
              MHB_TL_SPIN();
              v = ld_relaxed(pp);
            }
            prefix += v & kLbValueMask;
            if ((v & kLbStatusMask) == kLbInclusive || p == (u32)j) done = true;
          }
        }
        while (!done) {
          p -= LBW;
          u64 wv[LBW];
#pragma unroll
          for (int j = 0; j < LBW; ++j)
            wv[j] = (p >= (u32)j) ? ld_relaxed(lookback + (u64)(p - j) * 256 + tid) : 0ull;
#pragma unroll
          for (int j = 0; j < LBW; ++j) {
            if (!done) {
              u64 v = wv[j];
              const u64 *pp = lookback + (u64)(p - j) * 256 + tid;
              MHB_TL_DEPTH();
              while ((v & kLbStatusMask) == 0 || (v & lb_epoch(255)) != epv) {
                MHB_TL_SPIN();
                v = ld_relaxed(pp);
              }
              prefix += v & kLbValueMask;
              if ((v & kLbStatusMask) == kLbInclusive || p == (u32)j) done = true;
            }
          }
        }
        st_relaxed(lookback + (u64)tile * 256 + tid, kLbInclusive | epv | (prefix + (u64)pub));
      }
      s_glob[tid] = bin_addr[tid] + (prefix - (u64)excl) * (u64)(WR * 4);  // may address another GPU's memory
      MHB_TL_LB_DONE();
      MHB_TL_MARK(5);
    }
    __syncthreads();  // B4: s_recs and s_glob complete; nobody reads the counters any more
    MHB_TL_MARK(6);

    // ---- coalesced scatter + next digit's histogram; clear the counters for the next tile ----
    {
      uint4 *z = reinterpret_cast<uint4 *>(s_cnt);
      for (int i = tid; i < NW * 256 / 4; i += THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
      for (int i = tid; i < 256; i += THREADS) s_early[i] = 0;
    }
    const u64 my_off = (u64)tid * (WR * 4);
    if (full) {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const u32 p = (u32)i * THREADS + tid;
        u32 q[WR];
        ld_rec<WR>(s_recs, p, q);
        const u32 dd = rec_digit<WR>(q, widx, bsel);
        st_rec<WR>(reinterpret_cast<u32 *>(s_glob[dd] + my_off + (u64)i * (THREADS * WR * 4)), 0, q);
        if constexpr (HAS_NEXT) atomicAdd(&s_next[rec_digit<WR>(q, nwidx, nbsel)], 1u);
      }
    } else {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const u32 p = (u32)i * THREADS + tid;
        if (p < valid) {
          u32 q[WR];
          ld_rec<WR>(s_recs, p, q);
          const u32 dd = rec_digit<WR>(q, widx, bsel);
          st_rec<WR>(reinterpret_cast<u32 *>(s_glob[dd] + (u64)p * (WR * 4)), 0, q);
          if constexpr (HAS_NEXT) atomicAdd(&s_next[rec_digit<WR>(q, nwidx, nbsel)], 1u);
        }
      }
    }
    __syncthreads();  // B5: s_recs / s_glob free, counters zero
    MHB_TL_MARK(7);
    MHB_TL_FLUSH();
    tile = next_tile;
  }

  if constexpr (HAS_NEXT) {
    for (int i = tid; i < 256; i += THREADS)
      if (s_next[i]) atomicAdd((unsigned long long *)&next_hist[i], (unsigned long long)s_next[i]);
  }
}

}  // namespace mhb
