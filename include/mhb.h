/*
 * mhb.h -- C ABI of libmhb (megahit_b200): the B200-native SdBG-construction hot path of MEGAHIT.
 *
 * Plain pointers and sizes only; no C++ or torch types.  Status: 0 = ok, non-zero = error
 * (mhb_last_error() returns the message).  There is NO CPU fallback: every compute entry point fails
 * with MHB_ERR_CUDA when no CUDA device / kernel image is available.
 *
 * Reference interfaces replaced (paths relative to voutcn/megahit v1.2.9 src/):
 *   mhb_count_*     <- KmerCounter (sorting/kmer_counter.{h,cpp}) driven by main_kmer_count
 *                      (main_sdbg_build.cpp:35-86) through BaseSequenceSortingEngine::Run
 *                      (sorting/base_engine.cpp:143-211)
 *   mhb_sort_*      <- SelectSortingFunc / kmlib::kmsort (sorting/kmsort_selector.cpp:61-64,
 *                      kmlib/kmsort.h:43-122): sort fixed-width uint32 records by their leading words
 *   mhb_s2s_*       <- SeqToSdbg (sorting/seq_to_sdbg.{h,cpp}) driven by main_seq2sdbg
 *                      (main_sdbg_build.cpp:158-224)
 *   *_run           <- the `megahit_core count` / `megahit_core seq2sdbg` sub-commands themselves
 *                      (main.cpp:82-86), same option names and on-disk formats
 *
 * Layers:
 *   1. device level  -- raw device pointers + a cudaStream_t (as void*); the caller (PyTorch, or the
 *                       host pipeline below) owns all memory.  Used by tests, bench.py and the
 *                       multi-GPU driver (megahit_b200/multigpu.py).
 *   2. host level    -- host buffers in, host buffers out (H2D/D2H inside).
 *   3. file level    -- reads/writes the reference's on-disk formats; what `megahit_core` calls.
 */
#ifndef MHB_H
#define MHB_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MHB_OK 0
#define MHB_ERR_ARG 1
#define MHB_ERR_CUDA 2
#define MHB_ERR_IO 3
#define MHB_ERR_NOMEM 4

#define MHB_NUM_BUCKETS 65536 /* sorting/base_engine.h: kNumBuckets (8-base prefix) */
#define MHB_MAX_MUL 65535     /* sdbg/sdbg_def.h:12 kMaxMul */
#define MHB_MAX_K 255         /* sdbg/sdbg_def.h:20 kMaxK */
#define MHB_SENTINEL_OFFSET 0xFFFFFFFFu /* kmer_counter.h:49 */

const char *mhb_last_error(void);
const char *mhb_version(void);
/* number of visible CUDA devices (0 when none); never fails */
int mhb_device_count(void);
/* kernels launched by this process through libmhb so far (counted at every launch site; bench.py's gpu_launches) */
uint64_t mhb_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Geometry helpers (pure host arithmetic, callable without a GPU)
 * ------------------------------------------------------------------------------------------- */
/* words per `count` sort record on the device: the canonical (k+1)-mer left-aligned, then zero bits,
 * then prev<<3|next in the low 6 bits of the last word (the reference carries a 64-bit read_info
 * payload instead, kmer_counter.cpp:240-249; we re-derive read positions in mhb_count_mark_mercy). */
uint32_t mhb_count_record_words(uint32_t k);
/* words per edge in `.edges` files: ceil((2(k+1)+16)/32)  (kmer_counter.cpp:79-80) */
uint32_t mhb_words_per_edge(uint32_t k);
/* words per seq2sdbg sort record: ceil((2k+20)/32)  (seq_to_sdbg.cpp:510-512) */
uint32_t mhb_s2s_record_words(uint32_t k);
/* byte positions (0 = least significant byte of the last word) the LSD radix sort visits, ascending;
 * returns the count, at most 4*words. */
uint32_t mhb_count_sort_bytes(uint32_t k, uint8_t *bytes);
uint32_t mhb_s2s_sort_bytes(uint32_t k, uint8_t *bytes);
/* bytes of scratch mhb_sort_records needs for n records */
size_t mhb_sort_workspace_bytes(uint64_t n, uint32_t words);

/* ---------------------------------------------------------------------------------------------
 * 1. Device level.  All pointers are device pointers unless marked host.  `stream` is a cudaStream_t.
 * ------------------------------------------------------------------------------------------- */

/* A read library resident on the device in `.bin` layout (sequence_package.h:224-240): per read a
 * u32 length followed by ceil(len/16) words, forward (file) orientation.  The device code applies the
 * reversal that KmerCounter::Initialize does at load time (kmer_counter.cpp:61,72).
 * fixed_len > 0: every read has that length, record r starts at word r*(1+ceil(fixed_len/16));
 * rec_off/edge_off may then be NULL.  Otherwise rec_off[n_reads+1] gives each record's first word and
 * edge_off[n_reads+1] the exclusive prefix sum of max(0, len-k).
 * `bin` must be 16-byte aligned and its allocation padded to a multiple of 16 bytes. */
typedef struct {
  const uint32_t *bin;
  uint64_t bin_words;
  uint64_t n_reads;
  uint32_t fixed_len;
  const uint64_t *rec_off;
  const uint64_t *edge_off;
} mhb_dev_reads;

/* A1-A3: canonical (k+1)-mer extraction (kmer_counter.cpp:114-252).  Writes n_edges records of
 * mhb_count_record_words(k) words to `records` and adds the 256-bin histogram of record byte
 * `hist_byte` into hist256 (uint64[256], caller-zeroed; pass NULL to skip). */
int mhb_count_extract(void *stream, const mhb_dev_reads *reads, uint32_t k, uint32_t *records,
                      uint64_t n_edges, uint64_t *hist256, int hist_byte);

/* *flag_dev (device uint64, caller-zeroed) becomes non-zero when a read of a library handed over as fixed-length
 * (fixed_len > 0) has another length: the host-level calls look at a sample of the length words only and verify here. */
int mhb_check_fixed_len(void *stream, const uint32_t *bin_dev, uint64_t n_reads, uint32_t fixed_len, uint64_t *flag_dev);

/* A13 (base_engine.cpp:54-141, 254-281: Lv1 passes over bucket ranges): the same extraction restricted to the edges
 * whose 16-bit bucket id (first eight bases, kNumBuckets = 65536) lies in [lo, hi], for libraries whose records do
 * not fit in HBM at once.  Two calls per round: write = 0 fills per_read[0..n_reads] (device uint64) with the exclusive prefix of the
 * per-read in-range edge counts and *total_dev with their sum; write = 1 stores the in-range records compactly, in
 * read order, at records[per_read[r]...).  hist256 (optional, caller-zeroed) += histogram of record byte hist_byte
 * over the in-range records. */
int mhb_count_extract_range(void *stream, const mhb_dev_reads *reads, uint32_t k, uint32_t lo, uint32_t hi, int write,
                            uint64_t *per_read, uint32_t *records, uint64_t *hist256, int hist_byte,
                            uint64_t *total_dev);

/* A4: stable LSD radix sort of n records of `words` uint32 each, ascending on the given byte
 * positions (least significant first).  `first_hist` = histogram of bytes[0] if the caller already has
 * it (from mhb_count_extract / mhb_s2s_extract), else NULL.  Result is left in `a` if *result_in_b == 0
 * else in `b`.  ws = workspace of mhb_sort_workspace_bytes() bytes. */
int mhb_sort_records(void *stream, uint32_t *a, uint32_t *b, uint64_t n, uint32_t words,
                     const uint8_t *bytes, uint32_t n_bytes, const uint64_t *first_hist, void *ws,
                     size_t ws_bytes, int *result_in_b);

/* The same sort for callers that do not care in which order records with ALL sorted bytes equal come out (the count and
 * seq2sdbg stages: such records are tallied / reduced to their minimum multiplicity): the first pass may then be the
 * unstable partition pass (no look-back chain, one shared-memory atomic per record instead of stable ranking). */
int mhb_sort_records_relaxed(void *stream, uint32_t *a, uint32_t *b, uint64_t n, uint32_t words, const uint8_t *bytes,
                             uint32_t n_bytes, const uint64_t *first_hist, void *ws, size_t ws_bytes, int *result_in_b);

/* Fused partition + exchange for the multi-GPU path: ONE unstable radix pass whose per-digit destinations are arbitrary
 * device byte addresses (bin_addr_dev[256], device memory) = where the first record of digit d coming from THIS call
 * goes.  The digit of a record is owner_of_byte_dev[record byte `byte`] (256-entry device table mapping the record's
 * leading byte to the owning rank; required).  Digits owned by another GPU point into that GPU's receive buffer (opened
 * with mhb_ipc_open), so the scatter stores cross NVLink inside the partitioning kernel and no separate all-to-all is
 * needed.  The order of the records inside an owner's block is unspecified.  ws as for mhb_sort_records. */
int mhb_partition_scatter(void *stream, const uint32_t *recs, uint64_t n, uint32_t words, int byte,
                          const uint8_t *owner_of_byte_dev, const uint64_t *bin_addr_dev, void *ws, size_t ws_bytes);
/* The same pass, additionally delivering one histogram of record byte `next_byte` per owner (*hist_done = 1 on
 * success): owner_next_hist[o * 256 + v] (device uint64[16 * 256], caller-zeroed) += records sent to owner o whose byte
 * next_byte is v.  Summed over the sending ranks it is the
 * first-pass histogram of the owner's sort, which then need not sweep its records to count. */
int mhb_partition_scatter_hist(void *stream, const uint32_t *recs, uint64_t n, uint32_t words, int byte,
                               const uint8_t *owner_of_byte_dev, const uint64_t *bin_addr_dev, void *ws, size_t ws_bytes,
                               int next_byte, uint64_t *owner_next_hist, int *hist_done);
/* The bucket-range plan of one stage of the multi-GPU build, computed on the device from the all-gathered top-byte
 * histograms hist_all_dev[world][256] (so that nothing but a few counters has to visit the host between the histogram
 * exchange and the partition pass): rank r owns the leading-byte values [bounds[r], bounds[r+1]), cut where the
 * cumulative record count is closest to r/world of the total (canonical (k+1)-mers are A-skewed: equal-width ranges
 * would not balance).  Outputs, all device memory: owner_lut_dev[256] (leading byte -> owning rank),
 * bin_addr_dev[256] (entry o < world: byte address, inside owner o's receive buffer peer_base_host[o], where THIS
 * rank's block starts; for mhb_partition_scatter), plan_dev[64] = {[0..15] records owner o receives in total,
 * [16..31] records this rank sends to owner o, [32..32+world] bounds}.  world <= 16. */
int mhb_plan_partition(void *stream, const uint64_t *hist_all_dev, uint32_t world, uint32_t rank, uint32_t record_bytes,
                       const uint64_t *peer_base_host, uint8_t *owner_lut_dev, uint64_t *bin_addr_dev, uint64_t *plan_dev);
/* The solid edges with aux != 0 (the "tips" the mercy bookkeeping needs from every rank), compacted in no particular
 * order: tips_out gets records of mhb_words_per_edge(k) words, tip_aux_out their flags, *cursor_dev (device uint64,
 * caller-zeroed) ends at their number (entries beyond `capacity` are counted but not stored). */
int mhb_compact_tip_edges(void *stream, const uint32_t *edges, const uint8_t *aux, uint64_t n_solid, uint32_t k,
                          uint32_t *tips_out, uint8_t *tip_aux_out, uint64_t capacity, uint64_t *cursor_dev);
/* cudaMalloc'ed buffers that can be shared between the per-GPU processes of one node (CUDA IPC) */
int mhb_dev_malloc(void **ptr, size_t bytes);
int mhb_dev_free(void *ptr);
int mhb_ipc_export(const void *dev_ptr, uint8_t *handle64);
int mhb_ipc_open(const uint8_t *handle64, void **peer_ptr);
int mhb_ipc_close(void *peer_ptr);

/* Per-pass device times (ms, CUDA events on `stream`) of one of the last four sorts issued by this process:
 * back = 0 is the most recent.  Synchronises on that sort's last event only. */
int mhb_sort_pass_ms(int back, double *pass_ms, uint32_t max_passes, uint32_t *n_passes, uint64_t *n_records,
                     uint32_t *words);

/* A5/A6: run-length count over sorted records, solid filter, edge packing
 * (kmer_counter.cpp:254-381, PackEdge :32-52).
 *   edges_out   capacity_edges * mhb_words_per_edge(k) words, ascending solid edges
 *   aux_out     capacity_edges bytes: bit0 = no incoming, bit1 = no outgoing (for solid edges)
 *   mul_hist    uint64[65536], caller-zeroed: multiplicity histogram of ALL distinct edges
 *   n_solid_out device uint64 (caller-zeroed)
 *   scratch     mhb_count_solid_scratch_bytes(n) bytes
 * If the number of solid edges exceeds capacity_edges the surplus is not written; *n_solid_out still
 * reports the true count so the caller can retry. */
size_t mhb_count_solid_scratch_bytes(uint64_t n);
int mhb_count_solid(void *stream, const uint32_t *sorted_records, uint64_t n, uint32_t k, int32_t m,
                    uint32_t *edges_out, uint8_t *aux_out, uint64_t capacity_edges, uint64_t *mul_hist,
                    uint64_t *n_solid_out, void *scratch, size_t scratch_bytes);

/* A4 + A5 without the full sort, for 8-byte count records (11 <= k <= 28) and 1 <= m <= 1024: the records are grouped
 * by their leading 24 key bits with three radix passes (record bytes 5, 6, 7), cut into key-closed slices inside the
 * reference's 16-bit buckets, and every slice is aggregated by a hash table in shared memory - occurrence counts,
 * prev/next tallies of the keys that reach m, a counting sort of the slice's solid keys.  Same outputs, bit for bit,
 * as mhb_sort_records on all key bytes followed by mhb_count_solid, for under half of the memory traffic.  recs_a holds
 * the n extracted records (any order) and recs_b is a same-sized buffer; both are clobbered.  hist_byte5 = histogram
 * of record byte 5 (from mhb_count_extract) or NULL.  mul_hist / n_solid_out caller-zeroed as for mhb_count_solid.  ws = mhb_count_hashed_workspace_bytes(). */
int mhb_count_hashed_supported(uint32_t k, int32_t m);
size_t mhb_count_hashed_workspace_bytes(uint64_t n, uint32_t k, int32_t m);
int mhb_count_solid_hashed(void *stream, uint32_t *recs_a, uint32_t *recs_b, uint64_t n, uint32_t k, int32_t m,
                           const uint64_t *hist_byte5, uint32_t *edges_out, uint8_t *aux_out, uint64_t capacity_edges,
                           uint64_t *mul_hist, uint64_t *n_solid_out, void *ws, size_t ws_bytes);

/* A5 (mercy bookkeeping, kmer_counter.cpp:307-367): for every read, first_0_out / last_0_in exactly as
 * KmerCounter leaves them.  tips = hash set built by mhb_tipset_build from the solid edges whose aux
 * flags are non-zero. */
size_t mhb_tipset_bytes(uint64_t n_tip_edges, uint32_t k);
int mhb_tipset_build(void *stream, const uint32_t *edges, const uint8_t *aux, uint64_t n_solid, uint32_t k,
                     void *tipset, size_t tipset_bytes, uint64_t n_tip_edges);
int mhb_count_mark_mercy(void *stream, const mhb_dev_reads *reads, uint32_t k, const void *tipset,
                         size_t tipset_bytes, uint64_t n_tip_edges, uint32_t *first_0_out, uint32_t *last_0_in);
/* number of solid edges with aux != 0 (device reduction; result to host) */
int mhb_count_tip_edges(void *stream, const uint8_t *aux, uint64_t n_solid, uint64_t *n_tip_host);

/* A11 on the device (seq_to_sdbg.cpp:171-357 GenMercyEdges).
 * mhb_mercy_candidates: ascending ids of the reads KmerCounter would write to `.cand`
 *   (kmer_counter.cpp:390-401); cand_ids needs room for n_reads entries; *n_cand_host is set on return.
 * mhb_mercy_edges: the mercy (k+1)-mers of those reads, searched in the sorted solid `edges` (n_edges records of
 *   mhb_words_per_edge(k) words), written as `.edges`-format records with multiplicity 1 to mercy_out
 *   (capacity records), candidates in id order, positions ascending.  max_read_len bounds the reads' lengths. */
size_t mhb_mercy_candidates_scratch_bytes(uint64_t n_reads);
int mhb_mercy_candidates(void *stream, const uint32_t *first_0_out, const uint32_t *last_0_in, uint64_t n_reads,
                         uint64_t *cand_ids, uint64_t *n_cand_host, void *scratch, size_t scratch_bytes);
size_t mhb_mercy_edges_scratch_bytes(uint64_t n_cand, uint32_t max_read_len);
int mhb_mercy_edges(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                    uint32_t max_read_len, uint32_t k, const uint32_t *edges, uint64_t n_edges, uint32_t *mercy_out,
                    uint64_t capacity, uint64_t *n_mercy_host, void *scratch, size_t scratch_bytes);
/* The two halves of the search, for callers that size the destination from the exact count (the reference reserves
 * +25 % and grows, seq_to_sdbg.cpp:371-379): _count runs the probes and leaves per-read counts + offsets in `scratch`
 * (mhb_mercy_edges_scratch_bytes() minus mhb_edge_lut_bytes() bytes, luts built by the caller with mhb_edge_lut_build),
 * returning the number of mercy edges; _write emits exactly n_mercy records from the same, untouched scratch. */
int mhb_mercy_edges_count(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                          uint32_t max_read_len, uint32_t k, uint32_t n_segs, const uint32_t *const *seg_edges,
                          const uint64_t *seg_counts, const void *const *seg_luts, const uint8_t *owner_of_byte,
                          uint64_t *n_mercy_host, void *scratch, size_t scratch_bytes);
int mhb_mercy_edges_write(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                          uint32_t max_read_len, uint32_t k, uint32_t *mercy_out, uint64_t capacity, uint64_t n_mercy,
                          void *scratch, size_t scratch_bytes);

/* Multi-GPU form of the search (one process per GPU, each owning a contiguous range of leading bytes): every binary
 * search GenMercyEdges issues targets exactly one owner, and has_in / has_out are ORs over search outcomes, so each
 * rank answers - for the candidate reads of ALL ranks - the searches that land in its own range from local memory:
 * mhb_mercy_probe_owned writes 5 answer planes per read (mhb_mercy_planes_words() u32 words for n_cand reads;
 * cand_ids may be NULL = reads 0..n_cand-1), the ranks exchange planes, and mhb_mercy_count_planes ORs the n_src
 * planes of this rank's own candidates (source s at planes + s*src_stride_words), leaving scratch ready for
 * mhb_mercy_edges_write exactly as mhb_mercy_edges_count does. */
size_t mhb_mercy_planes_words(uint64_t n_cand, uint32_t max_read_len);
int mhb_mercy_probe_owned(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                          uint32_t max_read_len, uint32_t k, const uint32_t *edges, uint64_t n_edges, const void *lut,
                          const uint8_t *owner_of_byte, uint32_t me, uint32_t *planes_out);
int mhb_mercy_count_planes(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                           uint32_t max_read_len, uint32_t k, const uint32_t *planes, uint32_t n_src,
                           uint64_t src_stride_words, uint64_t *n_mercy_host, void *scratch, size_t scratch_bytes);

/* Same as mhb_mercy_edges, with the sorted solid edges given as n_segs (<= 16) segments: segment owner_of_byte[b] holds every edge whose
 * leading byte is b (host arrays; the segment pointers are device pointers and may be CUDA IPC peer pointers into
 * other GPUs' memory, so a multi-GPU build needs no gather of the edges). */
int mhb_mercy_edges_segs(void *stream, const mhb_dev_reads *reads, const uint64_t *cand_ids, uint64_t n_cand,
                         uint32_t max_read_len, uint32_t k, uint32_t n_segs, const uint32_t *const *seg_edges,
                         const uint64_t *seg_counts, const void *const *seg_luts, const uint8_t *owner_of_byte,
                         uint32_t *mercy_out, uint64_t capacity, uint64_t *n_mercy_host, void *scratch,
                         size_t scratch_bytes);
/* 12-base prefix -> [first,last] edge index table of one sorted edge segment (InitLookupTable, seq_to_sdbg.cpp:100-127);
 * mhb_edge_lut_bytes() bytes of device memory, one per segment, required by mhb_mercy_edges_segs. */
size_t mhb_edge_lut_bytes(void);
int mhb_edge_lut_build(void *stream, const uint32_t *edges, uint64_t n_edges, uint32_t k, void *lut);

/* Sequences in package orientation for seq2sdbg: word-aligned 2-bit packing.
 * fixed_len > 0: sequence s starts at word s*fixed_stride (fixed_stride = 0 means ceil(fixed_len/16));
 * word_off/len/item_off may be NULL.  With mult == NULL the multiplicity of sequence s is the low 16 bits
 * of the last word of its stride, i.e. `words` may be the `.edges` records themselves (edge_reader.h:49).
 * Otherwise word_off[n+1], len[n], item_off[n+1] (exclusive prefix of 2*(len-k+2) for len >= k+1, else 0). */
typedef struct {
  const uint32_t *words;
  uint64_t n_words;
  uint64_t n_seqs;
  uint32_t fixed_len;
  const uint64_t *word_off;
  const uint32_t *len;
  const uint64_t *item_off;
  const uint16_t *mult; /* per sequence */
  uint32_t fixed_stride;
} mhb_dev_seqs;

/* A8/A9 (seq_to_sdbg.cpp:530-700): all sort items of both strands. */
int mhb_s2s_extract(void *stream, const mhb_dev_seqs *seqs, uint32_t k, uint32_t *records, uint64_t n_items,
                    uint64_t *hist256, int hist_byte);

/* A8/A9 for `.edges` records that still carry the count stage's flags (aux[e] bit0 = no incoming, bit1 = no outgoing,
 * as mhb_count_solid writes them; edges n_with_aux .. n_edges-1, e.g. mercy edges appended behind the solid ones, have
 * none): the offset-0 / offset-2 ("$") items that SeqToSdbg::Lv2Postprocess is certain to discard (seq_to_sdbg.cpp:
 * 760-776: a solid edge enters / leaves the node - which is what has_in / has_out of kmer_counter.cpp:297-305 prove)
 * are not generated, so the sort and the emitter see about a third of the 6 * n_edges items and produce the same bytes.
 * Items are appended at records[*cursor_dev ...) (device uint64, caller-zeroed; ends at the item count, items beyond
 * `capacity` are not stored) in no particular order; hist256 += histogram of record byte hist_byte. */
int mhb_s2s_extract_edges_pruned(void *stream, const uint32_t *edges, const uint8_t *aux, uint64_t n_edges,
                                 uint64_t n_with_aux, uint32_t k, uint32_t *records, uint64_t capacity,
                                 uint64_t *cursor_dev, uint64_t *hist256, int hist_byte);

/* A13 for seq2sdbg (base_engine.cpp:254-281): the sort items whose 16-bit bucket id (first eight bases) lies in
 * [lo, hi].  records == NULL: count only - hist256 (caller-zeroed) += histogram of record byte hist_byte over the
 * in-range items.  Otherwise the in-range records are appended (in no particular order) at records[*cursor_dev ...);
 * cursor_dev (device uint64, caller-zeroed) ends at the number of in-range items; items beyond `capacity` are not
 * stored. */
int mhb_s2s_extract_range(void *stream, const mhb_dev_seqs *seqs, uint32_t k, uint32_t *records, uint64_t n_items,
                          uint32_t lo, uint32_t hi, uint64_t *cursor_dev, uint64_t capacity, uint64_t *hist256,
                          int hist_byte);

/* A10 (seq_to_sdbg.cpp:702-789 + sdbg_writer.cpp:25-58): SdBG item stream from sorted records.
 *   bytes_out     capacity_bytes; the variable-length item stream in sorted (= bucket) order
 *   bucket_table  uint64[65536*4] device: per bucket {byte offset, #items, #tips, #large_mul};
 *   totals        uint64[16] device: [0]=bytes [1]=items [2]=tips [3]=large_mul [4..12]=w counts [13]=ones in last
 *   scratch       mhb_s2s_emit_scratch_bytes(n, k) */
size_t mhb_s2s_emit_scratch_bytes(uint64_t n, uint32_t k);
int mhb_s2s_emit(void *stream, const uint32_t *sorted_records, uint64_t n, uint32_t k, uint8_t *bytes_out,
                 uint64_t capacity_bytes, uint64_t *bucket_table, uint64_t *totals, void *scratch,
                 size_t scratch_bytes);

/* The same emitter for the items of the 1-pass build (read2sdbg stage 2, read_to_sdbg_s2.cpp:521-614: identical
 * group logic, multiplicity = run length, already folded into the records by the caller).  label_fmt = 1: tip labels
 * carry the raw words of the reference's stage-2 record (flags nondollar<<3 | prev in the low 4 bits of word
 * ceil((2k+4)/32)-1, read_to_sdbg_s2.cpp:483-485, :602-606) instead of the seq2sdbg record's; 0 = mhb_s2s_emit. */
int mhb_s2s_emit_fmt(void *stream, const uint32_t *sorted_records, uint64_t n, uint32_t k, uint8_t *bytes_out,
                     uint64_t capacity_bytes, uint64_t *bucket_table, uint64_t *totals, void *scratch,
                     size_t scratch_bytes, int label_fmt);

/* ---------------------------------------------------------------------------------------------
 * 2. Host level (buffers in host memory; device 0 unless mhb_set_device was called)
 * ------------------------------------------------------------------------------------------- */
/* One process drives one GPU: call this before any compute entry point.  Selecting the same device again is a no-op;
 * switching after the first compute call fails with MHB_ERR_ARG (per-process arena, kernel attributes, caches). */
int mhb_set_device(int device);

typedef struct {
  uint32_t k;
  int32_t m;                /* solid threshold (-m / --min_kmer_frequency) */
  const uint32_t *bin;      /* host `.bin` image */
  uint64_t bin_words;
  uint64_t n_reads;
  int want_mercy;           /* compute first_0_out/last_0_in + candidate ids */
} mhb_count_args;

typedef struct {
  uint64_t n_edge_records;  /* (k+1)-mer occurrences processed */
  uint64_t n_solid;
  uint32_t words_per_edge;
  uint32_t *edges;          /* malloc'ed, n_solid * words_per_edge; free with mhb_free */
  uint64_t n_cand;
  uint64_t *cand_ids;       /* malloc'ed ascending read ids (kmer_counter.cpp:390-401) */
  uint64_t n_has_tips;
  int64_t counting[MHB_MAX_MUL + 1]; /* edge_counter.h:44-52 */
  double t_h2d_ms, t_extract_ms, t_sort_ms, t_count_ms, t_mercy_ms, t_d2h_ms, t_total_ms;
  uint32_t n_sort_passes;
  uint32_t n_rounds;        /* 1, or the number of leading-byte rounds when the records did not fit at once (A13) */
  double sort_pass_ms[64];
} mhb_count_result;

int mhb_count_host(const mhb_count_args *args, mhb_count_result *res);
/* A13 (base_engine.cpp:54-141 AdjustMemory): mhb_count_host runs in rounds over ranges of the leading record byte
 * when the records of the whole library do not fit in device memory; this caps a round at max_records_per_round
 * records regardless of memory (0 = derive from free device memory).  The result does not depend on the cap. */
int mhb_set_round_limit(uint64_t max_records_per_round);
/* the same cap for mhb_s2s_host, in sort items per round (independent of the count cap; 0 = derive from memory) */
int mhb_set_s2s_round_limit(uint64_t max_items_per_round);
/* The round planner itself (host only, no GPU needed): cuts the 256 leading-byte values, given their record counts,
 * into contiguous ranges [lo_out[i], hi_out[i]] of at most max_records records each (cf. Lv1FindEndBuckets,
 * base_engine.cpp:254-281).  Returns the number of ranges, or -1 (mhb_last_error) when one byte value alone
 * exceeds the cap.  lo_out / hi_out need room for 256 entries. */
int mhb_plan_rounds(const uint64_t *hist256, uint64_t max_records, uint32_t *lo_out, uint32_t *hi_out);
/* The planner the host rounds use: leading bytes as above, except that a leading byte holding more than max_records is
 * cut on its second byte, i.e. on the reference's own 16-bit bucket ids (base_engine.cpp:254-281) - canonical
 * (k+1)-mers are skewed towards A-prefixes and poly-A / low-complexity data more so.  sub_hist = 256 x 256 counts,
 * row b = histogram of the second byte among records with leading byte b (only rows of oversized bytes are read; NULL
 * when there are none).  Outputs ranges [lo16, hi16] of bucket ids tiling 0..65535 (room for cap_out entries); returns
 * their number, or -1 when a single bucket exceeds the cap. */
int mhb_plan_rounds16(const uint64_t *hist256, const uint64_t *sub_hist, uint64_t max_records, uint32_t *lo16_out,
                      uint32_t *hi16_out, uint32_t cap_out);

typedef struct {
  uint32_t k;
  const uint32_t *words;    /* host package-orientation sequences, word aligned */
  const uint64_t *word_off; /* n_seqs + 1 */
  const uint32_t *len;      /* n_seqs */
  const uint16_t *mult;     /* n_seqs */
  uint64_t n_seqs;
} mhb_s2s_args;

typedef struct {
  uint64_t n_records;
  uint64_t n_items, n_tips, n_large_mul, n_bytes;
  uint32_t words_per_tip_label;
  uint8_t *bytes;                                /* malloc'ed item stream, bucket order */
  uint64_t bucket_table[MHB_NUM_BUCKETS * 4];    /* {byte offset, items, tips, large_mul} */
  uint64_t w_count[9];
  uint64_t ones_in_last;
  double t_total_ms, t_extract_ms, t_sort_ms, t_emit_ms;
} mhb_s2s_result;

int mhb_s2s_host(const mhb_s2s_args *args, mhb_s2s_result *res);

/* Fused k_min build (SURVEY.md 8f N1): reads in, SdBG out, everything between stays in HBM.
 * count (extract + sort + solid edges + mercy bookkeeping) -> mercy edges (device, need_mercy) -> seq2sdbg
 * (extract + sort + emit) over solid + mercy edges.  Equivalent to `megahit_core count` followed by
 * `megahit_core seq2sdbg --input_prefix P [--need_mercy]` without the `.edges`/`.cand` round trip.
 * sdbg_out (optional, e.g. pinned memory) receives the item stream when it is large enough; otherwise the
 * stream is malloc'ed into res->bytes.  want_edges additionally returns what `count` writes to disk. */
typedef struct {
  uint32_t k;
  int32_t m;
  const uint32_t *bin;
  uint64_t bin_words;
  uint64_t n_reads;
  int32_t need_mercy;
  int32_t want_edges;
  uint8_t *sdbg_out;
  uint64_t sdbg_out_capacity;
} mhb_build_args;

typedef struct {
  uint64_t n_edge_records, n_solid, n_cand, n_mercy, n_sort_items;
  uint32_t words_per_edge, words_per_tip_label;
  uint64_t n_items, n_tips, n_large_mul, n_bytes;
  uint8_t *bytes;         /* == args->sdbg_out when that was used, else malloc'ed (mhb_free) */
  uint64_t *bucket_table; /* malloc'ed, 65536 x {byte offset, items, tips, large_mul} */
  uint64_t w_count[9];
  uint64_t ones_in_last;
  uint32_t *edges;        /* want_edges: malloc'ed n_solid * words_per_edge */
  uint64_t *cand_ids;     /* want_edges: malloc'ed n_cand */
  int64_t *counting;      /* want_edges: malloc'ed 65536 */
  double t_total_ms, t_h2d_ms, t_count_ms, t_mercy_ms, t_s2s_ms, t_d2h_ms;
} mhb_build_result;

/* A13: when the resident plan does not fit in device memory (cudaMalloc fails), or a round cap is set with
 * mhb_set_round_limit / mhb_set_s2s_round_limit, the same graph is built stage by stage - count in rounds over bucket
 * ranges -> mercy edges -> seq2sdbg in rounds - with the solid edges passing through host memory once; same outputs. */
int mhb_build_host(const mhb_build_args *args, mhb_build_result *res);

/* The 1-pass k_min build (main_read2sdbg, main_sdbg_build.cpp:88-156; `megahit --kmin-1pass`, and the route the driver
 * forces for --min-count 1, src/megahit:540-542): Read2SdbgS1 (read_to_sdbg_s1.cpp; only when m > 1) marks the solid
 * (k+1)-mer occurrences and the mercy candidates - with kmlib::kmsort's order among equal keys reproduced, because
 * stage 1 reads prev/next of a group's FIRST record for the whole group (:393-401) -, the mercy step of
 * Read2SdbgS2::Initialize (read_to_sdbg_s2.cpp:117-263, need_mercy) adds the (k+1)-mers between tips, Read2SdbgS2
 * builds the SdBG from the marked occurrences.  Same argument / result structs as mhb_build_host: want_edges is
 * ignored (this route writes no edges); res->counting (malloc'ed, 65536) = what stage 1 dumps to P.counting (zero for
 * m == 1), res->n_solid = distinct stage-2 items, t_count_ms / t_mercy_ms = bucket partition / kmsort emulation.
 * Stage 1 handles k <= 237 (records of at most 17 words); larger k with m > 1 returns MHB_ERR_ARG. */
int mhb_read2sdbg_host(const mhb_build_args *args, mhb_build_result *res);

/* `megahit_core iterate` (SURVEY.md 8f N2; main_iterate.cpp:117-221, iterate/contig_flank_index.h:16-221,
 * iterate/kmer_collector.h:37-79): the iterative edges for k + step - every (k+step+1)-mer of a read whose step+1
 * consecutive (k+1)-mers are all covered by contig flanks or their matched extensions - as ascending, unique `.edges`
 * records of mhb_words_per_edge(k + step) words with multiplicity 0 (the reference stores none: FlankInfo::mul is never
 * filled in; it writes the same set in hash-table order).  contigs: word-aligned 2-bit sequences in FILE orientation,
 * already filtered as AsyncContigReader does (contigs flagged kStandalone / kLoop discarded, async_sequence_reader.h:87);
 * bin: the read library image (`.bin`, file orientation, async_sequence_reader.h:51).  step even, 2 .. 28
 * (main_iterate.cpp:86); k + 1 <= 240 (flank records of at most 17 words).  res->edges: malloc'ed (mhb_free). */
typedef struct {
  uint32_t k, step;
  const uint32_t *contig_words;
  const uint64_t *contig_word_off; /* n_contigs + 1 */
  const uint32_t *contig_len;      /* n_contigs */
  uint64_t n_contigs;
  const uint32_t *bin;
  uint64_t bin_words;
  uint64_t n_reads;
} mhb_iterate_args;

typedef struct {
  uint64_t n_flanks;        /* distinct flank (k+1)-mers in the index */
  uint64_t n_aligned_reads; /* reads that yielded at least one edge */
  uint64_t n_candidates;    /* edges before the set semantics of KmerCollector */
  uint64_t n_edges;
  uint32_t words_per_edge;
  uint32_t *edges;
  double t_total_ms;
} mhb_iterate_result;

int mhb_iterate_host(const mhb_iterate_args *args, mhb_iterate_result *res);

/* A11 from host buffers (SeqToSdbg::GenMercyEdges, seq_to_sdbg.cpp:171-357, as `seq2sdbg --need_mercy` runs it between
 * loading `.edges` / `.cand` and the sort): edges = n_edges sorted `.edges`-format records, cand_bin = the `.cand` image
 * (`.bin` record format, reads in the reversed orientation KmerCounter wrote them, kmer_counter.cpp:387-401).
 * *mercy_out = malloc'ed n_mercy `.edges`-format records with multiplicity 1 (mhb_free). */
int mhb_mercy_host(uint32_t k, const uint32_t *edges, uint64_t n_edges, const uint32_t *cand_bin, uint64_t cand_words,
                   uint32_t **mercy_out, uint64_t *n_mercy_out, uint64_t *n_cand_reads_out);

void mhb_free(void *p);
/* drop the cached device arena (host-level entry points keep it between calls) */
int mhb_release(void);

/* ---------------------------------------------------------------------------------------------
 * 3. File level: the sub-commands.  Option names/meaning as main_sdbg_build.cpp:42-57 and :164-189.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  uint32_t k;
  int32_t m;
  double host_mem;
  int32_t num_cpu_threads;
  const char *read_lib_file;
  const char *output_prefix;
  int32_t mem_flag;
} mhb_count_opts;

typedef struct {
  double host_mem;
  uint32_t k;
  uint32_t k_from;
  int32_t num_cpu_threads;
  const char *contig;
  const char *bubble;
  const char *addi_contig;
  const char *local_contig;
  const char *input_prefix;
  const char *output_prefix;
  int32_t need_mercy;
  int32_t mem_flag;
} mhb_seq2sdbg_opts;

/* main_read2sdbg options (main_sdbg_build.cpp:95-111): those of `count` plus --need_mercy */
typedef struct {
  uint32_t k;
  int32_t m;
  double host_mem;
  int32_t num_cpu_threads;
  const char *read_lib_file;
  const char *output_prefix;
  int32_t mem_flag;
  int32_t need_mercy;
} mhb_read2sdbg_opts;

/* main_iterate options (main_iterate.cpp:57-72) */
typedef struct {
  const char *contig_file;
  const char *bubble_file;
  const char *read_file; /* the read library's `.bin` */
  int32_t num_cpu_threads;
  uint32_t k;
  uint32_t step;
  const char *output_prefix;
} mhb_iterate_opts;

int mhb_count_run(const mhb_count_opts *opts);
int mhb_seq2sdbg_run(const mhb_seq2sdbg_opts *opts);
/* writes P.edges.0 (ascending, unlike the reference's hash-table order) and P.edges.info (`is_sorted 0`, num_buckets 0) */
int mhb_iterate_run(const mhb_iterate_opts *opts);
/* writes P.sdbg.0, P.sdbg_info, P.counting (m > 1) and the (empty) P.mercy_cand.<i> temp files of the reference */
int mhb_read2sdbg_run(const mhb_read2sdbg_opts *opts);

/* `count` on n_gpus GPUs of this node (fixed-length read libraries; anything else, or n_gpus <= 1, runs mhb_count_run).
 * One worker process per GPU is forked; each takes a contiguous block of the reads, the records meet on the rank that
 * owns their leading byte (fused partition + exchange into CUDA-IPC peer buffers, SURVEY.md 8e), every rank counts its
 * bucket range, the mercy searches are answered by the owners of the searched prefixes, and - because the solid
 * edges are already on the devices - the k_min SdBG is built in the same run.  Files: rank r writes P.edges.<r> and
 * P.sdbg.<r>, rank 0 the merged P.edges.info (num_files = n_gpus, edge_io_meta.h:25-44), P.sdbg_info
 * (sdbg_meta.cpp:44-61), P.cand, P.counting, and the marker P.sdbg_fused ("k need_mercy n_gpus") that lets a following
 * `seq2sdbg --need_mercy --input_prefix P -o P` return at once instead of rebuilding the same graph.  The caller must not
 * have initialised CUDA in this process (the workers are forked). */
int mhb_count_run_multi(const mhb_count_opts *opts, int n_gpus);

/* ---------------------------------------------------------------------------------------------
 * Self-test hooks (host): build ONE sort record with the same __host__ __device__ code the kernels
 * run, so CPU-only tests can compare the bit arithmetic with the oracle.  Not a compute path.
 * ------------------------------------------------------------------------------------------- */
int mhb_selftest_count_record(const uint32_t *read_words, uint32_t nwords, uint32_t L, uint32_t k, uint32_t q,
                              uint32_t *rec_out, uint32_t *strand_out);
int mhb_selftest_count_records_roll(const uint32_t *read_words, uint32_t nwords, uint32_t L, uint32_t k, uint32_t q,
                                    uint64_t *rec4_out, uint32_t *strand4_out);
int mhb_selftest_s2s_record(const uint32_t *seq_words, uint32_t nwords, uint32_t L, uint32_t k, uint32_t strand,
                            uint32_t offset, uint32_t mult, uint32_t *rec_out);

/* read2sdbg building blocks on host arrays (same __host__ __device__ code as the kernels): stage-1 record e of a
 * package-orientation read (rec_out: key words + 2), stage-2 item (seq2sdbg layout) + palindrome flag, kmsort of one
 * bucket (records of nw + 2 words), stage-1 Lv2Postprocess over one sorted bucket of a fixed-length library, and the
 * mercy step of one read.  Bit arrays: bit i of word i/32. */
int mhb_selftest_r2s_s1_record(const uint32_t *pkg_words, uint32_t nwords, uint32_t L, uint32_t k, uint32_t e,
                               uint64_t base_off, uint32_t *rec_out);
int mhb_selftest_r2s_item(const uint32_t *pkg_words, uint32_t nwords, uint32_t L, uint32_t k, uint32_t i, uint32_t strand,
                          uint32_t type, uint32_t *rec_out, uint32_t *palindrome_out);
int mhb_selftest_kmsort(uint32_t *recs, uint64_t n, uint32_t nw);
/* the shared-memory form of the same sort (walk on tags, staged ranges of at most wcap records; 0 = device default), buckets above `cap` tags fall back to the in-place walk */
int mhb_selftest_kmsort_smem(uint32_t *recs, uint64_t n, uint32_t nw, uint32_t cap, uint32_t wcap);
int mhb_selftest_r2s_s1_group(const uint32_t *recs, uint64_t n, uint32_t k, int32_t m, uint32_t fixed_len, uint64_t n_reads,
                              int need_mercy, uint32_t *is_solid, uint32_t *no_in, uint32_t *no_out, uint32_t *any,
                              int64_t *counting);
/* `iterate` with the device code's __host__ __device__ building blocks driven serially on the host (CPU tests only) */
int mhb_selftest_iterate(const mhb_iterate_args *args, mhb_iterate_result *res);
int mhb_selftest_r2s_mercy_read(uint32_t fixed_len, uint64_t n_reads, uint64_t r, uint32_t k, const uint32_t *is_solid,
                                const uint32_t *no_in, const uint32_t *no_out, const uint32_t *any, uint32_t *mercy,
                                uint32_t *added_out);

#ifdef __cplusplus
}
#endif
#endif /* MHB_H */
