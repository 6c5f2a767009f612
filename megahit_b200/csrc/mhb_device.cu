// mhb_device.cu -- device-level C ABI (see include/mhb.h, layer 1): kernel launches on caller-owned
// device memory.  Built for sm_100a only; there is no host fallback.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "mhb.h"
#include "mhb_count.cuh"
#include "mhb_internal.h"
#include "mhb_mercy.cuh"
#include "mhb_s2s.cuh"
#include "mhb_common.cuh"

using namespace mhb;

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
int mhb_set_error(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
extern "C" const char *mhb_last_error(void) { return g_err; }
extern "C" const char *mhb_version(void) { return "megahit_b200 0.1 (sm_100a; formats of megahit v1.2.9)"; }
extern "C" int mhb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}
extern "C" void mhb_free(void *p) { free(p); }
unsigned long long g_mhb_launches = 0;
extern "C" uint64_t mhb_launch_count(void) { return g_mhb_launches; }


// ------------------------------------------------------------------------------------------------
// geometry
// ------------------------------------------------------------------------------------------------
extern "C" uint32_t mhb_count_record_words(uint32_t k) { return count_record_words(k); }
extern "C" uint32_t mhb_words_per_edge(uint32_t k) { return words_per_edge(k); }
extern "C" uint32_t mhb_s2s_record_words(uint32_t k) { return s2s_record_words(k); }

extern "C" uint32_t mhb_count_sort_bytes(uint32_t k, uint8_t *bytes) {
  // key = top 2(k+1) bits of the record: every byte that holds at least one key bit
  const u32 wr = count_record_words(k), total_bits = 32 * wr, key_bits = 2 * (k + 1);
  const u32 lo = (total_bits - key_bits) / 8;
  u32 n = 0;
  for (u32 b = lo; b < 4 * wr; ++b) bytes[n++] = (uint8_t)b;
  return n;
}
extern "C" uint32_t mhb_s2s_sort_bytes(uint32_t k, uint8_t *bytes) {
  // The reference sorts the whole record (seq_to_sdbg.cpp: no payload words).  The low 16 bits
  // (65535 - multiplicity) only decide which of several records with identical bases and flags comes first, and
  // the only use of that is "the first record of an (a,b) run carries the largest multiplicity" (:778-785); the
  // emit kernel takes the run's minimum instead, so those two bytes are not sorted.  Byte 2 holds the flag bits
  // 16..19 (prev char, non-dollar); all-zero bytes between the flags and the k-mer are skipped.
  const u32 w = s2s_record_words(k), total_bits = 32 * w, key_bits = 2 * k;
  const u32 lo = (total_bits - key_bits) / 8;
  u32 n = 0;
  for (u32 b = 2; b < 4 * w; ++b)
    if (b == 2 || b >= lo) bytes[n++] = (uint8_t)b;
  return n;
}

// ------------------------------------------------------------------------------------------------
// dispatch helpers
// ------------------------------------------------------------------------------------------------

static int g_sm_count = 0;
static int g_bound_device = -1;
int mhb_sm_count() {
  if (!g_sm_count) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev);
    if (g_sm_count <= 0) g_sm_count = 148;
    if (g_bound_device < 0) g_bound_device = dev;  // first compute call: the process stays on this device
  }
  return g_sm_count;
}

ReadsView make_reads_view(const mhb_dev_reads *r) {
  ReadsView v;
  v.bin = r->bin;
  v.bin_words = r->bin_words;
  v.n_reads = r->n_reads;
  v.fixed_len = r->fixed_len;
  v.fixed_stride = r->fixed_len ? 1 + div_ceil(r->fixed_len, 16) : 0;
  v.rec_off = r->rec_off;
  v.edge_off = r->edge_off;
  return v;
}

int check_reads(const mhb_dev_reads *r, uint32_t k) {
  if (!r || k < 1 || k > MHB_MAX_K) return mhb_set_error(MHB_ERR_ARG, "bad reads/k (k=%u)", k);
  if (r->n_reads && !r->bin) return mhb_set_error(MHB_ERR_ARG, "reads->bin is NULL");
  if (((uintptr_t)r->bin & 15) != 0) return mhb_set_error(MHB_ERR_ARG, "reads->bin must be 16-byte aligned");
  if (!r->fixed_len && r->n_reads && (!r->rec_off || !r->edge_off))
    return mhb_set_error(MHB_ERR_ARG, "variable-length reads need rec_off and edge_off");
  return MHB_OK;
}

// grow-only per-device scratch for block sums of scans issued from entry points that take no scratch argument
static int grow_scratch(size_t bytes, void **out) {
  static void *buf[64] = {nullptr};
  static size_t cap[64] = {0};
  int dev = 0;
  CK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return mhb_set_error(MHB_ERR_CUDA, "device index %d out of range", dev);
  if (cap[dev] < bytes) {
    CK(cudaDeviceSynchronize());
    if (buf[dev]) cudaFree(buf[dev]);
    buf[dev] = nullptr;
    cap[dev] = 0;
    const size_t want = (bytes + 4095) & ~(size_t)4095;
    CK(cudaMalloc(&buf[dev], want));
    cap[dev] = want;
  }
  *out = buf[dev];
  return MHB_OK;
}
static int scan64(cudaStream_t st, u64 *v, u64 n, u64 *total_dev, u64 *bsum);

// every read of a library assumed fixed-length really has that length: *flag_dev (device uint64, caller-zeroed) != 0
// when one does not (the host-level calls look at a sample of the length words only and verify here)
static __global__ void k_check_fixed_len(const u32 *__restrict__ bin, u64 n_reads, u32 stride, u32 L, unsigned long long *flag) {
  bool bad = false;
  for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += (u64)gridDim.x * blockDim.x) bad |= bin[r * stride] != L;
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1ull);
}
extern "C" int mhb_check_fixed_len(void *stream, const uint32_t *bin_dev, uint64_t n_reads, uint32_t fixed_len, uint64_t *flag_dev) {
  if (n_reads == 0) return MHB_OK;
  if (!bin_dev || !flag_dev || !fixed_len) return mhb_set_error(MHB_ERR_ARG, "bad arguments");
  k_check_fixed_len<<<mhb_sm_count() * 8, 256, 0, (cudaStream_t)stream>>>(bin_dev, n_reads, 1 + div_ceil(fixed_len, 16), fixed_len,
                                                                     (unsigned long long *)flag_dev);
  CK_LAUNCH();
  return MHB_OK;
}

// ------------------------------------------------------------------------------------------------
// count: extract
// ------------------------------------------------------------------------------------------------
extern "C" int mhb_count_extract(void *stream, const mhb_dev_reads *reads, uint32_t k, uint32_t *records,
                                 uint64_t n_edges, uint64_t *hist256, int hist_byte) {
  if (int rc = check_reads(reads, k)) return rc;
  if (reads->n_reads == 0 || n_edges == 0) return MHB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const ReadsView rv = make_reads_view(reads);
  const u32 W = count_key_words(k), WR = count_record_words(k);
  const u64 n_batches = (rv.n_reads + kReadsPerBatch - 1) / kReadsPerBatch;
  const int grid = (int)(n_batches < (u64)(sm_count() * 8) ? n_batches : (u64)(sm_count() * 8));
#define M(WW)                                                                                              \
  if (W == WW && WR == WW)                                                                                 \
    k_count_extract<WW, WW><<<grid, kExtractThreads, 0, st>>>(rv, k, records, hist256, hist_byte);         \
  else if (W == WW && WR == WW + 1)                                                                        \
    k_count_extract<WW, WW + 1><<<grid, kExtractThreads, 0, st>>>(rv, k, records, hist256, hist_byte);     \
  else
  MHB_FOR_W(M) return mhb_set_error(MHB_ERR_ARG, "unsupported k=%u", k);
#undef M
  CK_LAUNCH();
  return MHB_OK;
}

// A13: one round of the out-of-core count stage.  write == 0: per_read[r] <- in-range edge count of read r, then an
// in-place exclusive scan (per_read[n_reads] and *total_dev <- total); hist256 (optional) += histogram of byte
// hist_byte over the in-range records.  write != 0: per_read holds the scanned offsets; the in-range records go to
// records[per_read[r] ...) in read order and hist256 += histogram of hist_byte (the first sort digit).
extern "C" int mhb_count_extract_range(void *stream, const mhb_dev_reads *reads, uint32_t k, uint32_t lo, uint32_t hi,
                                       int write, uint64_t *per_read, uint32_t *records, uint64_t *hist256, int hist_byte,
                                       uint64_t *total_dev) {
  if (int rc = check_reads(reads, k)) return rc;
  if (lo > hi || hi > 65535) return mhb_set_error(MHB_ERR_ARG, "bad bucket range [%u, %u]", lo, hi);
  if (!per_read || (write && !records) || (!write && !total_dev)) return mhb_set_error(MHB_ERR_ARG, "null buffer");
  cudaStream_t st = (cudaStream_t)stream;
  if (reads->n_reads == 0) {
    if (!write) CK(cudaMemsetAsync(total_dev, 0, 8, st));
    return MHB_OK;
  }
  const ReadsView rv = make_reads_view(reads);
  const u32 W = count_key_words(k), WR = count_record_words(k);
  const u64 n_batches = (rv.n_reads + kReadsPerBatch - 1) / kReadsPerBatch;
  const int grid = (int)(n_batches < (u64)(sm_count() * 8) ? n_batches : (u64)(sm_count() * 8));
#define M2(WW, WRR)                                                                                                   \
  if (W == WW && WR == WRR) {                                                                                         \
    if (write)                                                                                                        \
      k_count_extract_range<WW, WRR, true><<<grid, kExtractThreads, 0, st>>>(rv, k, lo, hi, per_read, records, hist256, hist_byte); \
    else                                                                                                              \
      k_count_extract_range<WW, WRR, false><<<grid, kExtractThreads, 0, st>>>(rv, k, lo, hi, per_read, records, hist256, hist_byte); \
  } else
#define M(WW) M2(WW, WW) M2(WW, WW + 1)
  MHB_FOR_W(M) return mhb_set_error(MHB_ERR_ARG, "unsupported k=%u", k);
#undef M
#undef M2
  CK_LAUNCH();
  if (!write) {
    // three-phase scan (the block sums live in this device's small scratch): a single-CTA scan over all reads would
    // dominate a library that needs many rounds
    u64 *bsum = nullptr;
    if (int rc = grow_scratch(((rv.n_reads / kScanTile) + 2) * 8, (void **)&bsum)) return rc;
    if (int rc = scan64(st, per_read, rv.n_reads, total_dev, bsum)) return rc;
    CK(cudaMemcpyAsync(per_read + rv.n_reads, total_dev, 8, cudaMemcpyDeviceToDevice, st));
  }
  return MHB_OK;
}

// ------------------------------------------------------------------------------------------------
// count: solid edges
// ------------------------------------------------------------------------------------------------
extern "C" int mhb_count_solid(void *stream, const uint32_t *sorted_records, uint64_t n, uint32_t k, int32_t m,
                               uint32_t *edges_out, uint8_t *aux_out, uint64_t capacity_edges, uint64_t *mul_hist,
                               uint64_t *n_solid_out, void *scratch, size_t scratch_bytes) {
  if (k < 1 || k > MHB_MAX_K || !mul_hist || !n_solid_out) return mhb_set_error(MHB_ERR_ARG, "bad args");
  if (n == 0) return MHB_OK;
  const size_t need = mhb_count_solid_scratch_bytes(n);
  if (scratch_bytes < need) return mhb_set_error(MHB_ERR_ARG, "count scratch too small (%zu < %zu)", scratch_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  const u32 WR = count_record_words(k);
  {
    // v3: lane-blocked judge -> scan of chunk totals -> gather/pack (mhb_count.cuh)
#define M(WW)                                                                                                          \
  if (WR == WW) {                                                                                                      \
    constexpr int CH = 32 * count3_ipl(WW);                                                                            \
    const u64 n_chunks = (n + CH - 1) / CH;                                                                            \
    if (n_chunks >= (1ull << 32)) return mhb_set_error(MHB_ERR_ARG, "too many records for one count launch");          \
    const u64 n_sblk = (n_chunks + kScanTile - 1) / kScanTile;                                                         \
    char *p = (char *)scratch;                                                                                         \
    u32 *ticket = (u32 *)p;                                                                                            \
    p += 256;                                                                                                          \
    uint2 *solid_list = (uint2 *)p;                                                                                    \
    p += ((size_t)n_chunks * CH * 8 + 255) & ~(size_t)255;                                                             \
    u32 *chunk_count = (u32 *)p;                                                                                       \
    p += ((size_t)n_chunks * 4 + 255) & ~(size_t)255;                                                                  \
    u64 *chunk_off = (u64 *)p;                                                                                         \
    p += ((size_t)n_chunks * 8 + 255) & ~(size_t)255;                                                                  \
    u64 *bsum = (u64 *)p;                                                                                              \
    CK(cudaMemsetAsync(ticket, 0, 256, st));                                                                           \
    const size_t smem = (size_t)kCount3Warps * count3_warp_words(WW) * 4;                                              \
    static int bps = 0;                                                                                                \
    if (!bps) {                                                                                                        \
      CK(cudaFuncSetAttribute(k_count_lanes<WW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));             \
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_count_lanes<WW>, kCount3Warps * 32, smem));             \
      if (bps < 1) bps = 1;                                                                                            \
    }                                                                                                                  \
    u64 grid = (u64)sm_count() * bps;                                                                                  \
    if (grid > (n_chunks + kCount3Warps - 1) / kCount3Warps) grid = (n_chunks + kCount3Warps - 1) / kCount3Warps;      \
    k_count_lanes<WW><<<(unsigned)grid, kCount3Warps * 32, smem, st>>>(sorted_records, n, k, m, (u32)n_chunks, ticket,  \
                                                                      solid_list, chunk_count, mul_hist);             \
    CK_LAUNCH();                                                                                                       \
    k_scan32_sums<<<(unsigned)n_sblk, kScanThreads, 0, st>>>(chunk_count, n_chunks, bsum);                             \
    CK_LAUNCH();                                                                                                       \
    k_scan_u64<<<1, 1024, 0, st>>>(bsum, n_sblk, n_solid_out);                                                         \
    CK_LAUNCH();                                                                                                       \
    k_scan32_apply<<<(unsigned)n_sblk, kScanThreads, 0, st>>>(chunk_count, n_chunks, bsum, chunk_off);                 \
    CK_LAUNCH();                                                                                                       \
    u64 gw = (n_chunks + 7) / 8;                                                                                       \
    if (gw > (u64)sm_count() * 16) gw = (u64)sm_count() * 16;                                                          \
    k_count_write<WW><<<(unsigned)gw, 256, 0, st>>>(sorted_records, k, (u32)n_chunks, solid_list, chunk_count,         \
                                                    chunk_off, edges_out, aux_out, capacity_edges);                   \
  }
    MHB_FOR_WR(M)
#undef M
    CK_LAUNCH();
    return MHB_OK;
  }
  return mhb_set_error(MHB_ERR_ARG, "unsupported k=%u", k);
}

extern "C" size_t mhb_count_solid_scratch_bytes(uint64_t n) {
  // solid list (8 B per record slot, chunk-rounded) + per-chunk count/offset (chunks of >= 128 records) + slack
  return (size_t)(n + 1024) * 8 + (size_t)(n / 128 + 2) * 12 + (size_t)(n / 128 / kScanTile + 2) * 8 + 4096;
}

// ------------------------------------------------------------------------------------------------
// count: mercy bookkeeping
// ------------------------------------------------------------------------------------------------
extern "C" size_t mhb_tipset_bytes(uint64_t n_tip_edges, uint32_t k) {
  return 16 + tipset_filter_words(n_tip_edges) * 4 + tipset_capacity(n_tip_edges) * (size_t)(count_key_words(k) + 1) * 4;
}

// a few device words for scalar results, allocated once per device (cudaMallocAsync/cudaFreeAsync per call
// was measured to cost tens to hundreds of ms when most of HBM is already reserved)
static int small_scratch(unsigned long long **out) {
  static unsigned long long *buf[64] = {nullptr};
  int dev = 0;
  CK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return mhb_set_error(MHB_ERR_CUDA, "device index %d out of range", dev);
  if (!buf[dev]) CK(cudaMalloc((void **)&buf[dev], 256));
  *out = buf[dev];
  return MHB_OK;
}

extern "C" int mhb_count_tip_edges(void *stream, const uint8_t *aux, uint64_t n_solid, uint64_t *n_tip_host) {
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long *d = nullptr;
  *n_tip_host = 0;
  if (n_solid == 0) return MHB_OK;
  if (int rc = small_scratch(&d)) return rc;
  CK(cudaMemsetAsync(d, 0, 8, st));
  k_count_tips<<<sm_count() * 4, 256, 0, st>>>(aux, n_solid, d);
  CK_LAUNCH();
  CK(cudaMemcpyAsync(n_tip_host, d, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MHB_OK;
}

extern "C" int mhb_tipset_build(void *stream, const uint32_t *edges, const uint8_t *aux, uint64_t n_solid, uint32_t k,
                                void *tipset, size_t tipset_bytes, uint64_t n_tip_edges) {
  if (tipset_bytes < mhb_tipset_bytes(n_tip_edges, k)) return mhb_set_error(MHB_ERR_ARG, "tipset too small");
  cudaStream_t st = (cudaStream_t)stream;
  const u64 hdr[2] = {tipset_capacity(n_tip_edges), tipset_filter_words(n_tip_edges)};
  const u64 cap = hdr[0], fwords = hdr[1];
  CK(cudaMemsetAsync(tipset, 0, mhb_tipset_bytes(n_tip_edges, k), st));
  CK(cudaMemcpyAsync(tipset, hdr, 16, cudaMemcpyHostToDevice, st));
  if (n_solid == 0) return MHB_OK;
  u32 *filter = (u32 *)((char *)tipset + 16);
  u32 *table = filter + fwords;
  const u32 W = count_key_words(k);
  const u64 g = (n_solid + 255) / 256;
#define M(WW) \
  if (W == WW) k_tipset_insert<WW><<<(unsigned)g, 256, 0, st>>>(edges, aux, n_solid, k, filter, fwords, table, cap);
  MHB_FOR_W(M)
#undef M
  CK_LAUNCH();
  return MHB_OK;
}

// 8-byte records (W == 2 implies k + 1 >= 17) take the rolling record builder, 4 positions per lane, three of them by
// shifting: 6.5 vs 7.4 ms for the per-position kernel on the bench workload (profiles/r2a_bench_roll.json)
template <int W, int WR>
static void launch_mark_mercy(cudaStream_t st, int grid, const ReadsView &rv, u32 k, const u32 *filter, u64 fwords,
                              const u32 *table, u64 cap, u32 *first_0_out, u32 *last_0_in) {
  if constexpr (W == 2 && WR == 2) k_mark_mercy_roll<<<grid, 256, 0, st>>>(rv, k, filter, fwords, table, cap, first_0_out, last_0_in);
  else k_mark_mercy<W, WR><<<grid, 256, 0, st>>>(rv, k, filter, fwords, table, cap, first_0_out, last_0_in);
}

extern "C" int mhb_count_mark_mercy(void *stream, const mhb_dev_reads *reads, uint32_t k, const void *tipset,
                                    size_t tipset_bytes, uint64_t n_tip_edges, uint32_t *first_0_out,
                                    uint32_t *last_0_in) {
  if (int rc = check_reads(reads, k)) return rc;
  if (reads->n_reads == 0) return MHB_OK;
  if (tipset_bytes < mhb_tipset_bytes(n_tip_edges, k)) return mhb_set_error(MHB_ERR_ARG, "bad tipset");
  cudaStream_t st = (cudaStream_t)stream;
  const ReadsView rv = make_reads_view(reads);
  const u32 W = count_key_words(k), WR = count_record_words(k);
  const u64 cap = tipset_capacity(n_tip_edges), fwords = tipset_filter_words(n_tip_edges);
  const u32 *filter = (const u32 *)((const char *)tipset + 16);
  const u32 *table = filter + fwords;
  u64 g64 = (rv.n_reads + 7) / 8;
  if (g64 > (u64)sm_count() * 16) g64 = (u64)sm_count() * 16;
  const int grid = (int)g64;
#define M(WW)                                                                                                          \
  if (W == WW && WR == WW)                                                                                             \
    launch_mark_mercy<WW, WW>(st, grid, rv, k, filter, fwords, table, cap, first_0_out, last_0_in);                    \
  else if (W == WW && WR == WW + 1)                                                                                    \
    launch_mark_mercy<WW, WW + 1>(st, grid, rv, k, filter, fwords, table, cap, first_0_out, last_0_in);                \
  else
  MHB_FOR_W(M) return mhb_set_error(MHB_ERR_ARG, "unsupported k=%u", k);
#undef M
  CK_LAUNCH();
  return MHB_OK;
}

// ------------------------------------------------------------------------------------------------
// seq2sdbg
// ------------------------------------------------------------------------------------------------
static SeqsView make_seqs_view(const mhb_dev_seqs *s) {
  SeqsView v;
  v.words = s->words;
  v.n_words = s->n_words;
  v.n_seqs = s->n_seqs;
  v.fixed_len = s->fixed_len;
  v.word_off = s->word_off;
  v.len = s->len;
  v.item_off = s->item_off;
  v.mult = s->mult;
  v.fixed_stride = s->fixed_stride;
  return v;
}

extern "C" int mhb_s2s_extract(void *stream, const mhb_dev_seqs *seqs, uint32_t k, uint32_t *records,
                               uint64_t n_items, uint64_t *hist256, int hist_byte) {
  if (!seqs || k < 9 || k > MHB_MAX_K) return mhb_set_error(MHB_ERR_ARG, "kmer size must be >= 9 and <= 255");
  if (n_items == 0) return MHB_OK;
  if (!seqs->mult && !(seqs->fixed_len && seqs->fixed_stride))
    return mhb_set_error(MHB_ERR_ARG, "seqs->mult is NULL (only allowed for fixed-stride edge records)");
  if (!seqs->fixed_len && (!seqs->word_off || !seqs->len || !seqs->item_off))
    return mhb_set_error(MHB_ERR_ARG, "variable-length sequences need word_off, len and item_off");
  if (seqs->fixed_len && seqs->fixed_len < k + 1) return mhb_set_error(MHB_ERR_ARG, "fixed_len < k+1");
  cudaStream_t st = (cudaStream_t)stream;
  const SeqsView sv = make_seqs_view(seqs);
  const u32 W = s2s_record_words(k);
  if (seqs->fixed_len == k + 1 && seqs->fixed_stride && !seqs->mult && k + 1 <= 32 && k + 1 > 16 &&
      n_items == seqs->n_seqs * 6) {
    // `.edges` records of short (k+1)-mers: one thread per edge, 64-bit arithmetic
    u64 ge = (seqs->n_seqs + 255) / 256;
    if (ge > (u64)sm_count() * 32) ge = (u64)sm_count() * 32;
    if (W == 2) k_s2s_extract_edges<2><<<(unsigned)ge, 256, 0, st>>>(seqs->words, seqs->n_seqs, seqs->fixed_stride, k, records, hist256, hist_byte);
    else if (W == 3) k_s2s_extract_edges<3><<<(unsigned)ge, 256, 0, st>>>(seqs->words, seqs->n_seqs, seqs->fixed_stride, k, records, hist256, hist_byte);
    else return mhb_set_error(MHB_ERR_ARG, "internal: unexpected record width %u", W);
    CK_LAUNCH();
    return MHB_OK;
  }
  u64 g = (n_items + 255) / 256;
  if (g > (u64)sm_count() * 32) g = (u64)sm_count() * 32;
#define M(WW) \
  if (W == WW) k_s2s_extract<WW><<<(unsigned)g, 256, 0, st>>>(sv, k, records, n_items, hist256, hist_byte);
  MHB_FOR_WR(M)
#undef M
  CK_LAUNCH();
  return MHB_OK;
}

extern "C" int mhb_s2s_extract_edges_pruned(void *stream, const uint32_t *edges, const uint8_t *aux, uint64_t n_edges,
                                            uint64_t n_with_aux, uint32_t k, uint32_t *records, uint64_t capacity,
                                            uint64_t *cursor_dev, uint64_t *hist256, int hist_byte) {
  if (!edges || (!aux && n_with_aux) || !records || !cursor_dev || k < 9 || k > MHB_MAX_K || n_with_aux > n_edges)
    return mhb_set_error(MHB_ERR_ARG, "bad args");
  if (n_edges == 0) return MHB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const u32 W = s2s_record_words(k), WE = words_per_edge(k);
  u64 g = (n_edges + 255) / 256;
  if (g > (u64)sm_count() * 32) g = (u64)sm_count() * 32;
#define M(WW)                                                                                                        \
  if (W == WW)                                                                                                       \
    k_s2s_extract_edges_pruned<WW><<<(unsigned)g, 256, 0, st>>>(edges, aux, n_edges, n_with_aux, WE, k, records,       \
                                                               (unsigned long long *)cursor_dev, capacity, hist256, hist_byte);
  MHB_FOR_WR(M)
#undef M
  CK_LAUNCH();
  return MHB_OK;
}

// A13 for seq2sdbg: the items whose leading record byte lies in [lo, hi].  records == NULL counts only (hist256 +=
// histogram of record byte hist_byte over the in-range items); otherwise the in-range records are appended at
// records[*cursor_dev ...) (cursor_dev: device uint64, caller-zeroed; ends at the number of in-range items even when
// that exceeds `capacity`, in which case the surplus was not stored).
extern "C" int mhb_s2s_extract_range(void *stream, const mhb_dev_seqs *seqs, uint32_t k, uint32_t *records, uint64_t n_items,
                                     uint32_t lo, uint32_t hi, uint64_t *cursor_dev, uint64_t capacity, uint64_t *hist256,
                                     int hist_byte) {
  if (!seqs || k < 9 || k > MHB_MAX_K) return mhb_set_error(MHB_ERR_ARG, "kmer size must be >= 9 and <= 255");
  if (lo > hi || hi > 65535) return mhb_set_error(MHB_ERR_ARG, "bad bucket range [%u, %u]", lo, hi);
  if (records && !cursor_dev) return mhb_set_error(MHB_ERR_ARG, "cursor is NULL");
  if (n_items == 0) return MHB_OK;
  if (!seqs->mult && !(seqs->fixed_len && seqs->fixed_stride))
    return mhb_set_error(MHB_ERR_ARG, "seqs->mult is NULL (only allowed for fixed-stride edge records)");
  if (!seqs->fixed_len && (!seqs->word_off || !seqs->len || !seqs->item_off))
    return mhb_set_error(MHB_ERR_ARG, "variable-length sequences need word_off, len and item_off");
  if (seqs->fixed_len && seqs->fixed_len < k + 1) return mhb_set_error(MHB_ERR_ARG, "fixed_len < k+1");
  cudaStream_t st = (cudaStream_t)stream;
  const SeqsView sv = make_seqs_view(seqs);
  const u32 W = s2s_record_words(k);
  u64 g = (n_items + 255) / 256;
  if (g > (u64)sm_count() * 32) g = (u64)sm_count() * 32;
#define M(WW)                                                                                                        \
  if (W == WW)                                                                                                       \
    k_s2s_extract_range<WW><<<(unsigned)g, 256, 0, st>>>(sv, k, records, n_items, lo, hi, (unsigned long long *)cursor_dev, \
                                                         capacity, hist256, hist_byte);
  MHB_FOR_WR(M)
#undef M
  CK_LAUNCH();
  return MHB_OK;
}

// in-place exclusive scan of n u64 values (three phases, no serial chain); total -> *total_dev
static int scan64(cudaStream_t st, u64 *v, u64 n, u64 *total_dev, u64 *bsum) {
  const u64 nb = (n + kScanTile - 1) / kScanTile;
  k_scan64_sums<<<(unsigned)nb, kScanThreads, 0, st>>>(v, n, bsum);
  CK_LAUNCH();
  k_scan_u64<<<1, 1024, 0, st>>>(bsum, nb, total_dev);
  CK_LAUNCH();
  k_scan64_apply<<<(unsigned)nb, kScanThreads, 0, st>>>(v, n, bsum);
  CK_LAUNCH();
  return MHB_OK;
}

static u64 emit2_chunks(u64 n, u32 W) {
#define M(WW) \
  if (W == WW) return (n + emit2_chunk(WW) - 1) / emit2_chunk(WW);
  MHB_FOR_WR(M)
#undef M
  return 0;
}
static u32 emit2_chunk_records(u32 W) {
#define M(WW) \
  if (W == WW) return (u32)emit2_chunk(WW);
  MHB_FOR_WR(M)
#undef M
  return 0;
}

extern "C" size_t mhb_s2s_emit_scratch_bytes(uint64_t n, uint32_t k) {
  const u32 W = s2s_record_words(k);
  const u64 nc = emit2_chunks(n, W);
  return (size_t)MHB_NUM_BUCKETS * (4 * 8 + 5 * 4) + (size_t)nc * 4 * (4 + 8) + (size_t)(nc / kScanTile + 2) * 8 +
         (size_t)nc * emit2_chunk_records(W) * emit2_max_item_bytes(k) + 4096;
}

extern "C" int mhb_s2s_emit(void *stream, const uint32_t *sorted_records, uint64_t n, uint32_t k, uint8_t *bytes_out,
                            uint64_t capacity_bytes, uint64_t *bucket_table, uint64_t *totals, void *scratch,
                            size_t scratch_bytes) {
  return mhb_s2s_emit_fmt(stream, sorted_records, n, k, bytes_out, capacity_bytes, bucket_table, totals, scratch,
                          scratch_bytes, 0);
}

extern "C" int mhb_s2s_emit_fmt(void *stream, const uint32_t *sorted_records, uint64_t n, uint32_t k, uint8_t *bytes_out,
                                uint64_t capacity_bytes, uint64_t *bucket_table, uint64_t *totals, void *scratch,
                                size_t scratch_bytes, int label_fmt) {
  const u32 fmt = label_fmt ? 1u : 0u;
  if (k < 9 || k > MHB_MAX_K || !bucket_table || !totals) return mhb_set_error(MHB_ERR_ARG, "bad args");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMemsetAsync(totals, 0, 16 * 8, st));
  CK(cudaMemsetAsync(bucket_table, 0, (size_t)MHB_NUM_BUCKETS * 4 * 8, st));
  if (n == 0) return MHB_OK;
  if (scratch_bytes < mhb_s2s_emit_scratch_bytes(n, k)) return mhb_set_error(MHB_ERR_ARG, "emit scratch too small");
  const u32 W = s2s_record_words(k);
  const u64 nc = emit2_chunks(n, W);
  if (nc >= (1ull << 32)) return mhb_set_error(MHB_ERR_ARG, "too many records for one emit launch");
  const u32 chrec = emit2_chunk_records(W), maxb = emit2_max_item_bytes(k);
  char *p = (char *)scratch;
  u64 *bucket_start = (u64 *)p;
  p += (size_t)MHB_NUM_BUCKETS * 4 * 8;
  u32 *bucket_local = (u32 *)p;
  p += (size_t)MHB_NUM_BUCKETS * 5 * 4;
  u64 *chunk_off = (u64 *)p;
  p += (size_t)nc * 4 * 8;
  u64 *bsum = (u64 *)p;
  p += (size_t)(nc / kScanTile + 2) * 8;
  u32 *chunk_tot = (u32 *)p;
  p += ((size_t)nc * 4 * 4 + 255) & ~(size_t)255;
  uint8_t *tmp = (uint8_t *)p;
  CK(cudaMemsetAsync(bucket_local, 0xFF, (size_t)MHB_NUM_BUCKETS * 5 * 4, st));
#define M(WW)                                                                                                       \
  if (W == WW) {                                                                                                    \
    const size_t smem = (size_t)kEmit2Warps * emit2_slots(WW) * WW * 4;                                             \
    static int bps = 0;                                                                                             \
    if (!bps) {                                                                                                     \
      CK(cudaFuncSetAttribute(k_s2s_judge<WW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));            \
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_s2s_judge<WW>, kEmit2Warps * 32, smem));             \
      if (bps < 1) bps = 1;                                                                                         \
    }                                                                                                               \
    u64 grid = (u64)sm_count() * bps;                                                                               \
    if (grid > (nc + kEmit2Warps - 1) / kEmit2Warps) grid = (nc + kEmit2Warps - 1) / kEmit2Warps;                   \
    k_s2s_judge<WW><<<(unsigned)grid, kEmit2Warps * 32, smem, st>>>(sorted_records, n, k, (u32)nc, tmp, chunk_tot,   \
                                                                   bucket_local, totals, fmt);                     \
  }
  MHB_FOR_WR(M)
#undef M
  CK_LAUNCH();
  for (int q = 0; q < 4; ++q)
    if (int rc = scan32(st, chunk_tot + (u64)q * nc, nc, chunk_off + (u64)q * nc, totals + q, bsum)) return rc;
  u64 gg = (nc + 7) / 8;
  if (gg > (u64)sm_count() * 16) gg = (u64)sm_count() * 16;
  k_s2s_gather<<<(unsigned)gg, 256, 0, st>>>(tmp, chrec, maxb, (u32)nc, chunk_tot, chunk_off, bytes_out, capacity_bytes);
  CK_LAUNCH();
  k_bucket_starts<<<64, 256, 0, st>>>(bucket_local, chunk_off, nc, bucket_start);
  CK_LAUNCH();
  k_bucket_finalize<<<1, 1024, 0, st>>>(bucket_start, totals, bucket_table);
  CK_LAUNCH();
  return MHB_OK;
}

// ------------------------------------------------------------------------------------------------
// mercy edges on the device (A11)
// ------------------------------------------------------------------------------------------------
int scan32(cudaStream_t st, const u32 *in, u64 n, u64 *out, u64 *total_dev, u64 *bsum) {
  const u64 nb = (n + kScanTile - 1) / kScanTile;
  k_scan32_sums<<<(unsigned)nb, kScanThreads, 0, st>>>(in, n, bsum);
  CK_LAUNCH();
  k_scan_u64<<<1, 1024, 0, st>>>(bsum, nb, total_dev);
  CK_LAUNCH();
  k_scan32_apply<<<(unsigned)nb, kScanThreads, 0, st>>>(in, n, bsum, out);
  CK_LAUNCH();
  return MHB_OK;
}

extern "C" size_t mhb_mercy_candidates_scratch_bytes(uint64_t n_reads) {
  return (size_t)(n_reads + 64) * 12 + (size_t)(n_reads / kScanTile + 2) * 8 + 1024;
}

extern "C" int mhb_mercy_candidates(void *stream, const uint32_t *first_0_out, const uint32_t *last_0_in,
                                    uint64_t n_reads, uint64_t *cand_ids, uint64_t *n_cand_host, void *scratch,
                                    size_t scratch_bytes) {
  *n_cand_host = 0;
  if (n_reads == 0) return MHB_OK;
  if (scratch_bytes < mhb_mercy_candidates_scratch_bytes(n_reads)) return mhb_set_error(MHB_ERR_ARG, "scratch too small");
  cudaStream_t st = (cudaStream_t)stream;
  char *p = (char *)scratch;
  u64 *total = (u64 *)p;
  p += 256;
  u32 *flag = (u32 *)p;
  p += ((size_t)n_reads * 4 + 255) & ~(size_t)255;
  u64 *off = (u64 *)p;
  p += ((size_t)n_reads * 8 + 255) & ~(size_t)255;
  u64 *bsum = (u64 *)p;
  const unsigned g = (unsigned)((n_reads + 255) / 256);
  k_cand_flags<<<g, 256, 0, st>>>(first_0_out, last_0_in, n_reads, flag);
  CK_LAUNCH();
  if (int rc = scan32(st, flag, n_reads, off, total, bsum)) return rc;
  k_cand_compact<<<g, 256, 0, st>>>(flag, off, n_reads, cand_ids);
  CK_LAUNCH();
  CK(cudaMemcpyAsync(n_cand_host, total, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MHB_OK;
}

extern "C" size_t mhb_edge_lut_bytes(void);
size_t mercy_core_scratch(uint64_t n_cand, uint32_t max_read_len) {
  const size_t wpr = (max_read_len + 31) / 32 + 1;
  return (size_t)n_cand * 3 * wpr * 4 + (size_t)(n_cand + 64) * 12 + (size_t)(n_cand / kScanTile + 2) * 8 + 2048;
}
// scratch for mhb_mercy_edges (single segment: includes room for its look-up table); the segmented call needs
// this minus mhb_edge_lut_bytes()
extern "C" size_t mhb_mercy_edges_scratch_bytes(uint64_t n_cand, uint32_t max_read_len) {
  return ((mercy_core_scratch(n_cand, max_read_len) + 255) & ~(size_t)255) + 512 + mhb_edge_lut_bytes();
}

extern "C" size_t mhb_edge_lut_bytes(void) { return (size_t)kLutEntries * sizeof(uint2); }

extern "C" int mhb_edge_lut_build(void *stream, const uint32_t *edges, uint64_t n_edges, uint32_t k, void *lut) {
  if (n_edges >= 0xFFFFFFFFull) return mhb_set_error(MHB_ERR_ARG, "too many edges for the 32-bit look-up table");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMemsetAsync(lut, 0xFF, mhb_edge_lut_bytes(), st));
  if (n_edges == 0) return MHB_OK;
  u64 g = (n_edges + 255) / 256;
  if (g > (u64)sm_count() * 16) g = (u64)sm_count() * 16;
  k_edge_lut<<<(unsigned)g, 256, 0, st>>>(edges, n_edges, words_per_edge(k), (uint2 *)lut);
  CK_LAUNCH();
  return MHB_OK;
}

MercyScratch mercy_scratch_layout(void *scratch, uint64_t n_cand, uint32_t max_read_len) {
  MercyScratch m;
  m.wpr = (max_read_len + 31) / 32 + 1;
  char *p = (char *)scratch;
  m.total = (u64 *)p;
  p += 256;
  m.bits = (u32 *)p;
  p += ((size_t)n_cand * 3 * m.wpr * 4 + 255) & ~(size_t)255;
  m.count = (u32 *)p;
  p += ((size_t)n_cand * 4 + 255) & ~(size_t)255;
  m.off = (u64 *)p;
  p += ((size_t)n_cand * 8 + 255) & ~(size_t)255;
  m.bsum = (u64 *)p;
  return m;
}

extern "C" int mhb_mercy_edges_count(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                                     uint32_t max_read_len, uint32_t k, uint32_t n_segs, const uint32_t *const *seg_edges,
                                     const uint64_t *seg_counts, const void *const *seg_luts, const uint8_t *owner_of_byte,
                                     uint64_t *n_mercy_host, void *scratch, size_t scratch_bytes) {
  *n_mercy_host = 0;
  if (int rc = check_reads(reads, k)) return rc;
  if (n_cand == 0) return MHB_OK;
  if (k < 12) return mhb_set_error(MHB_ERR_ARG, "mercy edges need k >= 12 (12-mer look-up prefix)");
  if (n_segs < 1 || n_segs > 16) return mhb_set_error(MHB_ERR_ARG, "1..16 edge segments supported");
  if (scratch_bytes < mercy_core_scratch(n_cand, max_read_len)) return mhb_set_error(MHB_ERR_ARG, "scratch too small");
  cudaStream_t st = (cudaStream_t)stream;
  const ReadsView rv = make_reads_view(reads);
  EdgeSegs sg;
  memset(&sg, 0, sizeof(sg));
  for (u32 i = 0; i < n_segs; ++i) {
    sg.ptr[i] = seg_edges[i];
    sg.n[i] = (long long)seg_counts[i];
    sg.lut[i] = (const uint2 *)seg_luts[i];
    if (!sg.lut[i]) return mhb_set_error(MHB_ERR_ARG, "segment %u has no look-up table (mhb_edge_lut_build)", i);
  }
  for (int b = 0; b < 256; ++b) {
    sg.owner[b] = owner_of_byte ? owner_of_byte[b] : 0;
    if (sg.owner[b] >= n_segs) return mhb_set_error(MHB_ERR_ARG, "owner_of_byte[%d] = %u out of range", b, sg.owner[b]);
  }
  const u32 WE = words_per_edge(k), WM = div_ceil(k + 1, 16);
  const MercyScratch ms = mercy_scratch_layout(scratch, n_cand, max_read_len);
  u64 g64 = (n_cand + 7) / 8;
  if (g64 > (u64)sm_count() * 16) g64 = (u64)sm_count() * 16;
#define M(WW) \
  if (WM == WW) k_mercy_probe<WW><<<(unsigned)g64, 256, 0, st>>>(rv, cand_ids, n_cand, k, sg, WE, ms.bits, ms.wpr);
  MHB_FOR_W(M)
#undef M
  CK_LAUNCH();
  const unsigned g = (unsigned)((n_cand + 127) / 128);
  k_mercy_emit<false><<<g, 128, 0, st>>>(rv, cand_ids, n_cand, k, ms.bits, ms.wpr, ms.count, nullptr, nullptr, WE);
  CK_LAUNCH();
  if (int rc = scan32(st, ms.count, n_cand, ms.off, ms.total, ms.bsum)) return rc;
  CK(cudaMemcpyAsync(n_mercy_host, ms.total, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MHB_OK;
}

extern "C" int mhb_mercy_edges_write(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                                     uint32_t max_read_len, uint32_t k, uint32_t *mercy_out, uint64_t capacity,
                                     uint64_t n_mercy, void *scratch, size_t scratch_bytes) {
  if (int rc = check_reads(reads, k)) return rc;
  if (n_cand == 0 || n_mercy == 0) return MHB_OK;
  if (scratch_bytes < mercy_core_scratch(n_cand, max_read_len)) return mhb_set_error(MHB_ERR_ARG, "scratch too small");
  if (n_mercy > capacity) return mhb_set_error(MHB_ERR_NOMEM, "mercy edges (%llu) exceed capacity (%llu)",
                                               (unsigned long long)n_mercy, (unsigned long long)capacity);
  cudaStream_t st = (cudaStream_t)stream;
  const ReadsView rv = make_reads_view(reads);
  const MercyScratch ms = mercy_scratch_layout(scratch, n_cand, max_read_len);
  const unsigned g = (unsigned)((n_cand + 127) / 128);
  k_mercy_emit<true><<<g, 128, 0, st>>>(rv, cand_ids, n_cand, k, ms.bits, ms.wpr, ms.count, ms.off, mercy_out, words_per_edge(k));
  CK_LAUNCH();
  return MHB_OK;
}

extern "C" int mhb_mercy_edges_segs(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                                    uint32_t max_read_len, uint32_t k, uint32_t n_segs, const uint32_t *const *seg_edges,
                                    const uint64_t *seg_counts, const void *const *seg_luts, const uint8_t *owner_of_byte,
                                    uint32_t *mercy_out, uint64_t capacity, uint64_t *n_mercy_host, void *scratch,
                                    size_t scratch_bytes) {
  if (int rc = mhb_mercy_edges_count(stream, reads, cand_ids, n_cand, max_read_len, k, n_segs, seg_edges, seg_counts, seg_luts,
                                     owner_of_byte, n_mercy_host, scratch, scratch_bytes))
    return rc;
  return mhb_mercy_edges_write(stream, reads, cand_ids, n_cand, max_read_len, k, mercy_out, capacity, *n_mercy_host, scratch,
                               scratch_bytes);
}

extern "C" int mhb_mercy_edges(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                               uint32_t max_read_len, uint32_t k, const uint32_t *edges, uint64_t n_edges,
                               uint32_t *mercy_out, uint64_t capacity, uint64_t *n_mercy_host, void *scratch,
                               size_t scratch_bytes) {
  *n_mercy_host = 0;
  if (n_cand == 0) return MHB_OK;
  // single segment: the look-up table lives behind the core scratch in the caller's buffer
  const size_t core = (mercy_core_scratch(n_cand, max_read_len) + 255) & ~(size_t)255;
  if (scratch_bytes < core + mhb_edge_lut_bytes()) return mhb_set_error(MHB_ERR_ARG, "scratch too small");
  void *lut = (char *)scratch + core;
  if (int rc = mhb_edge_lut_build(stream, edges, n_edges, k, lut)) return rc;
  const void *luts[1] = {lut};
  return mhb_mercy_edges_segs(stream, reads, cand_ids, n_cand, max_read_len, k, 1, &edges, &n_edges, luts, nullptr, mercy_out,
                              capacity, n_mercy_host, scratch, core);
}

// One process drives one GPU (the multi-GPU build is one process per GPU): kernel attributes, occupancy caches and the
// host-level arena are per process, so the device can be chosen once, before the first compute call; choosing the same
// device again is a no-op, switching afterwards is refused instead of silently dereferencing the other GPU's memory.
extern "C" int mhb_set_device(int device) {
  if (g_bound_device >= 0 && device != g_bound_device)
    return mhb_set_error(MHB_ERR_ARG, "this process is bound to CUDA device %d: mhb_set_device(%d) must be the first libmhb call "
                         "(one process per GPU)", g_bound_device, device);
  CK(cudaSetDevice(device));
  g_bound_device = device;
  g_sm_count = 0;
  return MHB_OK;
}
