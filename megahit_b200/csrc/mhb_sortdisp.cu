// mhb_sortdisp.cu -- the radix-sort part of the device-level C ABI (include/mhb.h, layer 1): per-width dispatch of the
// radix pass kernels (mhb_sort3.cuh = stable sort pass, mhb_part.cuh = unstable first pass and exchange pass), the
// fused partition + exchange pass, CUDA-IPC buffer helpers and the per-pass timing trace.  Its own translation unit
// because the kernel instantiations (17 record widths) dominate the build time of the library.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "mhb.h"
#include "mhb_common.cuh"
#include "mhb_kernels.cuh"
#include "mhb_sort.cuh"
#include "mhb_sort3.cuh"
#include "mhb_part.cuh"

using namespace mhb;

// ------------------------------------------------------------------------------------------------
// sort
// ------------------------------------------------------------------------------------------------
template <int WR>
static u64 sort_tiles(u64 n) {
  return (n + SortCfg3<WR>::TILE - 1) / SortCfg3<WR>::TILE;
}
static u64 sort_num_tiles(u64 n, u32 words) {
#define M(WW) \
  if (words == WW) return sort_tiles<WW>(n);
  MHB_FOR_WR(M)
#undef M
  return 0;
}
static constexpr size_t kSortHeadBytes = (size_t)(72 + 1) * 256 * 8 /*hist*/ + 256 * 8 /*bin_base*/ + 128 * 4 + 256 * 8 /*gcursor*/;

// head + the look-back descriptors of the stable pass: 256 64-bit descriptors per tile
extern "C" size_t mhb_sort_workspace_bytes(uint64_t n, uint32_t words) {
  return kSortHeadBytes + (size_t)sort_num_tiles(n, words) * 256 * 8 + 256;
}

template <int WR>
static int launch_radix_pass(cudaStream_t st, const u32 *in, u64 n, int byte_idx, const u64 *bin_base, u64 *lookback,
                             u32 *tile_counter, u64 *next_hist, int next_byte, u32 epoch) {
  using C = SortCfg3<WR>;
  static int blocks_per_sm = 0;
  if (!blocks_per_sm) {
    CK(cudaFuncSetAttribute(k_radix_pass3<WR, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    CK(cudaFuncSetAttribute(k_radix_pass3<WR, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, k_radix_pass3<WR, true>, C::THREADS, C::SMEM));
    if (blocks_per_sm < 1) return mhb_set_error(MHB_ERR_CUDA, "radix pass kernel (WR=%d) does not fit an SM", WR);
    if (getenv("MHB_VERBOSE")) fprintf(stderr, "[mhb] radix pass WR=%d: %d threads x %d rec, %zu B smem, %d CTA/SM\n", WR, C::THREADS, C::IPT, C::SMEM, blocks_per_sm);
  }
  const u64 tiles = sort_tiles<WR>(n);
  u64 grid = (u64)blocks_per_sm * sm_count();
  if (grid > tiles) grid = tiles;
  if (next_hist)
    k_radix_pass3<WR, true><<<(int)grid, C::THREADS, C::SMEM, st>>>(in, n, (u32)tiles, byte_idx, bin_base, lookback, tile_counter,
                                                                    next_hist, next_byte, epoch);
  else
    k_radix_pass3<WR, false><<<(int)grid, C::THREADS, C::SMEM, st>>>(in, n, (u32)tiles, byte_idx, bin_base, lookback, tile_counter,
                                                                     nullptr, 0, epoch);
  CK_LAUNCH();
  return MHB_OK;
}

// unstable pass (mhb_part.cuh): the first pass of a sort whose caller does not need a deterministic order among fully
// equal keys (OWNER_LUT = false), and the exchange pass, whose digit is the owning rank (OWNER_LUT = true)
template <int WR, bool OWNER_LUT>
static int launch_part_unstable(cudaStream_t st, const u32 *in, u64 n, int byte_idx, const u64 *bin_base,
                                unsigned long long *gcursor, u32 *tile_counter, u64 *next_hist, int next_byte,
                                const uint8_t *lut) {
  using C = PartCfg<WR>;
  constexpr size_t SMEM_HIST = OWNER_LUT ? C::SMEM_OWNER_HIST : C::SMEM;
  static int bps = 0;
  if (!bps) {
    CK(cudaFuncSetAttribute(k_part_unstable<WR, OWNER_LUT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_HIST));
    CK(cudaFuncSetAttribute(k_part_unstable<WR, OWNER_LUT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_part_unstable<WR, OWNER_LUT, true>, C::THREADS, SMEM_HIST));
    if (bps < 1) return mhb_set_error(MHB_ERR_CUDA, "partition pass (WR=%d) does not fit an SM", WR);
    if (getenv("MHB_VERBOSE")) fprintf(stderr, "[mhb] unstable partition pass WR=%d owner=%d: %d threads x %d rec, %zu B smem, %d CTA/SM\n", WR, (int)OWNER_LUT, C::THREADS, C::IPT, SMEM_HIST, bps);
  }
  const u64 tiles = (n + C::TILE - 1) / C::TILE;
  u64 grid = (u64)bps * sm_count();
  if (grid > tiles) grid = tiles;
  if (next_hist)
    k_part_unstable<WR, OWNER_LUT, true><<<(int)grid, C::THREADS, SMEM_HIST, st>>>(in, n, (u32)tiles, byte_idx, bin_base, gcursor,
                                                                                   tile_counter, next_hist, next_byte, lut);
  else
    k_part_unstable<WR, OWNER_LUT, false><<<(int)grid, C::THREADS, C::SMEM, st>>>(in, n, (u32)tiles, byte_idx, bin_base, gcursor,
                                                                                  tile_counter, nullptr, 0, lut);
  CK_LAUNCH();
  return MHB_OK;
}

#ifdef MHB_SORT_TIMELINE
// diagnostic build only: point the v3 radix pass at a device buffer of rows x 16 uint64 (see mhb_sort3.cuh)
extern "C" int mhb_debug_set_sort_timeline(unsigned long long *dev_buf, unsigned long long rows) {
  CK(cudaMemcpyToSymbol(g_sort_timeline, &dev_buf, sizeof(dev_buf)));
  CK(cudaMemcpyToSymbol(g_sort_timeline_rows, &rows, sizeof(rows)));
  return MHB_OK;
}
#endif

// Per-pass timing: every sort records one event before and after each pass into a small ring, so a
// caller can ask afterwards (mhb_sort_pass_ms) how long each pass of a recent sort took without putting a
// synchronisation inside its timed region.
namespace {
struct SortTrace {
  cudaEvent_t ev[74];
  bool created = false;
  uint32_t n_passes = 0, words = 0;
  uint64_t n = 0;
};
SortTrace g_trace[4];
uint64_t g_trace_seq = 0;
}  // namespace

// relaxed != 0: the first pass may be the unstable partition pass (mhb_part.cuh) - the order among records whose sorted
// bytes are ALL equal is then unspecified
int mhb_sort_records_ex(void *stream, uint32_t *a, uint32_t *b, uint64_t n, uint32_t words, const uint8_t *bytes,
                        uint32_t n_bytes, const uint64_t *first_hist, void *ws, size_t ws_bytes, int *result_in_b,
                        double *pass_ms_host, int relaxed);
int mhb_sort_records_impl(void *stream, uint32_t *a, uint32_t *b, uint64_t n, uint32_t words, const uint8_t *bytes,
                          uint32_t n_bytes, const uint64_t *first_hist, void *ws, size_t ws_bytes, int *result_in_b,
                          double *pass_ms_host) {
  // the library's own stages tally or minimise over records with equal sort keys: their order is irrelevant
  return mhb_sort_records_ex(stream, a, b, n, words, bytes, n_bytes, first_hist, ws, ws_bytes, result_in_b, pass_ms_host, 1);
}
int mhb_sort_records_ex(void *stream, uint32_t *a, uint32_t *b, uint64_t n, uint32_t words, const uint8_t *bytes,
                          uint32_t n_bytes, const uint64_t *first_hist, void *ws, size_t ws_bytes, int *result_in_b,
                        double *pass_ms_host, int relaxed) {
  if (words < 1 || words > 17 || n_bytes > 72 || !result_in_b)
    return mhb_set_error(MHB_ERR_ARG, "bad sort geometry (words=%u n_bytes=%u)", words, n_bytes);
  *result_in_b = 0;
  if (n == 0 || n_bytes == 0) return MHB_OK;
  if (ws_bytes < mhb_sort_workspace_bytes(n, words)) return mhb_set_error(MHB_ERR_ARG, "sort workspace too small");
  if (n >= (1ull << 53)) return mhb_set_error(MHB_ERR_ARG, "too many records");
  cudaStream_t st = (cudaStream_t)stream;
  u64 *hist = (u64 *)ws;                        // [n_bytes+1][256]
  u64 *bin_base = hist + (72 + 1) * 256;        // [256]
  u32 *tile_counter = (u32 *)(bin_base + 256);  // [128]
  unsigned long long *gcursor = (unsigned long long *)(tile_counter + 128);  // [256]: unstable first pass
  u64 *lookback = (u64 *)((char *)ws + kSortHeadBytes);
  CK(cudaMemsetAsync(ws, 0, mhb_sort_workspace_bytes(n, words), st));
  if (first_hist) {
    CK(cudaMemcpyAsync(hist, first_hist, 256 * 8, cudaMemcpyDeviceToDevice, st));
  } else {
#define M(WW) \
  if (words == WW) k_hist_byte<WW><<<sm_count() * 4, 256, 0, st>>>(a, n, bytes[0], hist);
    MHB_FOR_WR(M)
#undef M
    CK_LAUNCH();
  }
  SortTrace &tr = g_trace[g_trace_seq++ & 3];
  if (!tr.created) {
    for (int i = 0; i < 74; ++i) CK(cudaEventCreate(&tr.ev[i]));
    tr.created = true;
  }
  tr.n_passes = n_bytes;
  tr.words = words;
  tr.n = n;
  CK(cudaEventRecord(tr.ev[0], st));
  u32 *in = a, *out = b;
  for (u32 p = 0; p < n_bytes; ++p) {
    k_hist_scan256<<<1, 256, 0, st>>>(hist + (u64)p * 256, bin_base, (u64)(uintptr_t)out, words * 4);
    CK_LAUNCH();
    u64 *next_hist = p + 1 < n_bytes ? hist + (u64)(p + 1) * 256 : nullptr;
    const int next_byte = p + 1 < n_bytes ? bytes[p + 1] : 0;
    int rc = MHB_ERR_ARG;
    if (p == 0 && relaxed && words == 2) rc = launch_part_unstable<2, false>(st, in, n, bytes[p], bin_base, gcursor, tile_counter + p, next_hist, next_byte, nullptr);
    else if (p == 0 && relaxed && words == 3) rc = launch_part_unstable<3, false>(st, in, n, bytes[p], bin_base, gcursor, tile_counter + p, next_hist, next_byte, nullptr);
    else {
#define M(WW) \
  if (words == WW) rc = launch_radix_pass<WW>(st, in, n, bytes[p], bin_base, lookback, tile_counter + p, next_hist, next_byte, p + 1);
      MHB_FOR_WR(M)
#undef M
    }
    if (rc) return rc;
    CK(cudaEventRecord(tr.ev[p + 1], st));
    u32 *t = in;
    in = out;
    out = t;
  }
  *result_in_b = (in == b) ? 1 : 0;
  if (pass_ms_host) {
    CK(cudaEventSynchronize(tr.ev[n_bytes]));
    for (u32 p = 0; p < n_bytes; ++p) {
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, tr.ev[p], tr.ev[p + 1]));
      pass_ms_host[p] = ms;
    }
  }
  return MHB_OK;
}

// ------------------------------------------------------------------------------------------------
// fused partition + exchange: one radix pass whose per-digit destinations are arbitrary device addresses, e.g.
// slots inside OTHER GPUs' receive buffers opened through CUDA IPC.  The scatter stores travel over NVLink while
// the rest of the tile is still being ranked - no separate all-to-all.  The exchange has no earlier order to preserve
// (every receiving stage re-sorts and tallies, or takes the minimum over equal keys), so it is the unstable pass.
// ------------------------------------------------------------------------------------------------
static int partition_scatter_impl(void *stream, const uint32_t *recs, uint64_t n, uint32_t words, int byte,
                                  const uint8_t *owner_of_byte_dev, const uint64_t *bin_addr_dev, void *ws, size_t ws_bytes,
                                  int next_byte, uint64_t *owner_next_hist) {
  if (!owner_of_byte_dev) return mhb_set_error(MHB_ERR_ARG, "owner table is NULL");
  if (words < 1 || words > 17 || byte < 0 || byte >= (int)(4 * words)) return mhb_set_error(MHB_ERR_ARG, "bad geometry");
  if (n == 0) return MHB_OK;
  if (ws_bytes < kSortHeadBytes) return mhb_set_error(MHB_ERR_ARG, "sort workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  u32 *tile_counter = (u32 *)((u64 *)ws + (72 + 1) * 256 + 256);
  unsigned long long *gcursor = (unsigned long long *)(tile_counter + 128);
  CK(cudaMemsetAsync(ws, 0, kSortHeadBytes, st));
  int rc = MHB_ERR_ARG;
#define M(WW)                                                                                                          \
  if (words == WW)                                                                                                     \
    rc = launch_part_unstable<WW, true>(st, recs, n, byte, bin_addr_dev, gcursor, tile_counter, owner_next_hist, next_byte, \
                                        owner_of_byte_dev);
  MHB_FOR_WR(M)
#undef M
  return rc;
}
extern "C" int mhb_partition_scatter(void *stream, const uint32_t *recs, uint64_t n, uint32_t words, int byte,
                                     const uint8_t *owner_of_byte_dev, const uint64_t *bin_addr_dev, void *ws,
                                     size_t ws_bytes) {
  return partition_scatter_impl(stream, recs, n, words, byte, owner_of_byte_dev, bin_addr_dev, ws, ws_bytes, 0, nullptr);
}
extern "C" int mhb_partition_scatter_hist(void *stream, const uint32_t *recs, uint64_t n, uint32_t words, int byte,
                                          const uint8_t *owner_of_byte_dev, const uint64_t *bin_addr_dev, void *ws,
                                          size_t ws_bytes, int next_byte, uint64_t *owner_next_hist, int *hist_done) {
  if (!owner_of_byte_dev || !owner_next_hist || !hist_done || next_byte < 0 || next_byte >= (int)(4 * words))
    return mhb_set_error(MHB_ERR_ARG, "bad owner-histogram arguments");
  *hist_done = 0;
  if (int rc = partition_scatter_impl(stream, recs, n, words, byte, owner_of_byte_dev, bin_addr_dev, ws, ws_bytes, next_byte,
                                      owner_next_hist))
    return rc;
  *hist_done = 1;
  return MHB_OK;
}

extern "C" int mhb_dev_malloc(void **ptr, size_t bytes) {
  CK(cudaMalloc(ptr, bytes));
  return MHB_OK;
}
extern "C" int mhb_dev_free(void *ptr) {
  CK(cudaFree(ptr));
  return MHB_OK;
}
extern "C" int mhb_ipc_export(const void *dev_ptr, uint8_t *handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, const_cast<void *>(dev_ptr)));
  memcpy(handle64, &h, 64);
  return MHB_OK;
}
extern "C" int mhb_ipc_open(const uint8_t *handle64, void **peer_ptr) {
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  CK(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return MHB_OK;
}
extern "C" int mhb_ipc_close(void *peer_ptr) {
  CK(cudaIpcCloseMemHandle(peer_ptr));
  return MHB_OK;
}

extern "C" int mhb_sort_pass_ms(int back, double *pass_ms, uint32_t max_passes, uint32_t *n_passes, uint64_t *n_records,
                                uint32_t *words) {
  if (back < 0 || back > 3 || (uint64_t)back >= g_trace_seq) return mhb_set_error(MHB_ERR_ARG, "no such sort in the trace ring");
  SortTrace &tr = g_trace[(g_trace_seq - 1 - back) & 3];
  CK(cudaEventSynchronize(tr.ev[tr.n_passes]));
  for (u32 p = 0; p < tr.n_passes && p < max_passes; ++p) {
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, tr.ev[p], tr.ev[p + 1]));
    pass_ms[p] = ms;
  }
  if (n_passes) *n_passes = tr.n_passes;
  if (n_records) *n_records = tr.n;
  if (words) *words = tr.words;
  return MHB_OK;
}

extern "C" int mhb_sort_records(void *stream, uint32_t *a, uint32_t *b, uint64_t n, uint32_t words,
                                const uint8_t *bytes, uint32_t n_bytes, const uint64_t *first_hist, void *ws,
                                size_t ws_bytes, int *result_in_b) {
  return mhb_sort_records_ex(stream, a, b, n, words, bytes, n_bytes, first_hist, ws, ws_bytes, result_in_b, nullptr, 0);
}

extern "C" int mhb_sort_records_relaxed(void *stream, uint32_t *a, uint32_t *b, uint64_t n, uint32_t words,
                                        const uint8_t *bytes, uint32_t n_bytes, const uint64_t *first_hist, void *ws,
                                        size_t ws_bytes, int *result_in_b) {
  return mhb_sort_records_ex(stream, a, b, n, words, bytes, n_bytes, first_hist, ws, ws_bytes, result_in_b, nullptr, 1);
}

