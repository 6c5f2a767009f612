"""ctypes binding of libmhb.so (the C ABI declared in include/mhb.h).

This is the host-side mirror of the reference's interface for the SdBG-construction path:
`count_run` / `seq2sdbg_run` take the same options as `megahit_core count` / `seq2sdbg`
(src/main_sdbg_build.cpp:42-57, :164-189), `count_host` / `s2s_host` are the in-memory equivalents of
KmerCounter::Run / SeqToSdbg::Run, and the `dev_*` functions are the individual device stages working
on torch tensors (device memory, streams = plumbing).

There is NO CPU fallback: every compute entry point raises MhbError when the CUDA library or a device
is missing.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# MHB_LIB selects another build of the same library (e.g. libmhb_timeline.so, the diagnostic build); never a fallback
LIB_PATH = os.environ.get("MHB_LIB") or os.path.join(_HERE, "libmhb.so")
NUM_BUCKETS = 65536
SENTINEL_OFFSET = 0xFFFFFFFF

_lib = None


class MhbError(RuntimeError):
    pass


class DevReads(C.Structure):
    _fields_ = [("bin", C.c_void_p), ("bin_words", C.c_uint64), ("n_reads", C.c_uint64), ("fixed_len", C.c_uint32),
                ("rec_off", C.c_void_p), ("edge_off", C.c_void_p)]


class DevSeqs(C.Structure):
    _fields_ = [("words", C.c_void_p), ("n_words", C.c_uint64), ("n_seqs", C.c_uint64), ("fixed_len", C.c_uint32),
                ("word_off", C.c_void_p), ("len", C.c_void_p), ("item_off", C.c_void_p), ("mult", C.c_void_p),
                ("fixed_stride", C.c_uint32)]


class CountArgs(C.Structure):
    _fields_ = [("k", C.c_uint32), ("m", C.c_int32), ("bin", C.c_void_p), ("bin_words", C.c_uint64),
                ("n_reads", C.c_uint64), ("want_mercy", C.c_int)]


class CountResult(C.Structure):
    _fields_ = [("n_edge_records", C.c_uint64), ("n_solid", C.c_uint64), ("words_per_edge", C.c_uint32),
                ("edges", C.POINTER(C.c_uint32)), ("n_cand", C.c_uint64), ("cand_ids", C.POINTER(C.c_uint64)),
                ("n_has_tips", C.c_uint64), ("counting", C.c_int64 * 65536),
                ("t_h2d_ms", C.c_double), ("t_extract_ms", C.c_double), ("t_sort_ms", C.c_double),
                ("t_count_ms", C.c_double), ("t_mercy_ms", C.c_double), ("t_d2h_ms", C.c_double),
                ("t_total_ms", C.c_double), ("n_sort_passes", C.c_uint32), ("n_rounds", C.c_uint32), ("sort_pass_ms", C.c_double * 64)]


class S2sArgs(C.Structure):
    _fields_ = [("k", C.c_uint32), ("words", C.c_void_p), ("word_off", C.c_void_p), ("len", C.c_void_p),
                ("mult", C.c_void_p), ("n_seqs", C.c_uint64)]


class S2sResult(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_items", C.c_uint64), ("n_tips", C.c_uint64),
                ("n_large_mul", C.c_uint64), ("n_bytes", C.c_uint64), ("words_per_tip_label", C.c_uint32),
                ("bytes", C.POINTER(C.c_uint8)), ("bucket_table", C.c_uint64 * (65536 * 4)),
                ("w_count", C.c_uint64 * 9), ("ones_in_last", C.c_uint64),
                ("t_total_ms", C.c_double), ("t_extract_ms", C.c_double), ("t_sort_ms", C.c_double),
                ("t_emit_ms", C.c_double)]


class BuildArgs(C.Structure):
    _fields_ = [("k", C.c_uint32), ("m", C.c_int32), ("bin", C.c_void_p), ("bin_words", C.c_uint64),
                ("n_reads", C.c_uint64), ("need_mercy", C.c_int32), ("want_edges", C.c_int32),
                ("sdbg_out", C.c_void_p), ("sdbg_out_capacity", C.c_uint64)]


class BuildResult(C.Structure):
    _fields_ = [("n_edge_records", C.c_uint64), ("n_solid", C.c_uint64), ("n_cand", C.c_uint64), ("n_mercy", C.c_uint64),
                ("n_sort_items", C.c_uint64), ("words_per_edge", C.c_uint32), ("words_per_tip_label", C.c_uint32),
                ("n_items", C.c_uint64), ("n_tips", C.c_uint64), ("n_large_mul", C.c_uint64), ("n_bytes", C.c_uint64),
                ("bytes", C.POINTER(C.c_uint8)), ("bucket_table", C.POINTER(C.c_uint64)), ("w_count", C.c_uint64 * 9),
                ("ones_in_last", C.c_uint64), ("edges", C.POINTER(C.c_uint32)), ("cand_ids", C.POINTER(C.c_uint64)),
                ("counting", C.POINTER(C.c_int64)),
                ("t_total_ms", C.c_double), ("t_h2d_ms", C.c_double), ("t_count_ms", C.c_double),
                ("t_mercy_ms", C.c_double), ("t_s2s_ms", C.c_double), ("t_d2h_ms", C.c_double)]


class CountOpts(C.Structure):
    _fields_ = [("k", C.c_uint32), ("m", C.c_int32), ("host_mem", C.c_double), ("num_cpu_threads", C.c_int32),
                ("read_lib_file", C.c_char_p), ("output_prefix", C.c_char_p), ("mem_flag", C.c_int32)]


class Seq2SdbgOpts(C.Structure):
    _fields_ = [("host_mem", C.c_double), ("k", C.c_uint32), ("k_from", C.c_uint32), ("num_cpu_threads", C.c_int32),
                ("contig", C.c_char_p), ("bubble", C.c_char_p), ("addi_contig", C.c_char_p),
                ("local_contig", C.c_char_p), ("input_prefix", C.c_char_p), ("output_prefix", C.c_char_p),
                ("need_mercy", C.c_int32), ("mem_flag", C.c_int32)]


class Read2SdbgOpts(C.Structure):
    _fields_ = [("k", C.c_uint32), ("m", C.c_int32), ("host_mem", C.c_double), ("num_cpu_threads", C.c_int32),
                ("read_lib_file", C.c_char_p), ("output_prefix", C.c_char_p), ("mem_flag", C.c_int32),
                ("need_mercy", C.c_int32)]


class IterateArgs(C.Structure):
    _fields_ = [("k", C.c_uint32), ("step", C.c_uint32), ("contig_words", C.c_void_p), ("contig_word_off", C.c_void_p),
                ("contig_len", C.c_void_p), ("n_contigs", C.c_uint64), ("bin", C.c_void_p), ("bin_words", C.c_uint64),
                ("n_reads", C.c_uint64)]


class IterateResult(C.Structure):
    _fields_ = [("n_flanks", C.c_uint64), ("n_aligned_reads", C.c_uint64), ("n_candidates", C.c_uint64), ("n_edges", C.c_uint64),
                ("words_per_edge", C.c_uint32), ("edges", C.POINTER(C.c_uint32)), ("t_total_ms", C.c_double)]


class IterateOpts(C.Structure):
    _fields_ = [("contig_file", C.c_char_p), ("bubble_file", C.c_char_p), ("read_file", C.c_char_p),
                ("num_cpu_threads", C.c_int32), ("k", C.c_uint32), ("step", C.c_uint32), ("output_prefix", C.c_char_p)]


# every symbol include/mhb.h declares (tests/test_abi.py checks the header against this list)
SYMBOLS = [
    "mhb_last_error", "mhb_version", "mhb_device_count", "mhb_launch_count", "mhb_count_record_words", "mhb_words_per_edge",
    "mhb_s2s_record_words", "mhb_count_sort_bytes", "mhb_s2s_sort_bytes", "mhb_sort_workspace_bytes",
    "mhb_count_extract", "mhb_check_fixed_len", "mhb_count_extract_range", "mhb_set_round_limit", "mhb_set_s2s_round_limit", "mhb_plan_rounds", "mhb_plan_rounds16", "mhb_sort_records", "mhb_sort_records_relaxed", "mhb_sort_pass_ms", "mhb_partition_scatter", "mhb_partition_scatter_hist", "mhb_plan_partition", "mhb_compact_tip_edges", "mhb_dev_malloc", "mhb_dev_free",
    "mhb_ipc_export", "mhb_ipc_open", "mhb_ipc_close", "mhb_count_solid_scratch_bytes", "mhb_count_solid", "mhb_count_hashed_supported", "mhb_count_hashed_workspace_bytes", "mhb_count_solid_hashed", "mhb_tipset_bytes",
    "mhb_tipset_build", "mhb_count_mark_mercy", "mhb_count_tip_edges", "mhb_s2s_extract", "mhb_s2s_extract_range",
    "mhb_s2s_emit_scratch_bytes", "mhb_s2s_emit", "mhb_set_device", "mhb_count_host", "mhb_s2s_host", "mhb_build_host", "mhb_free",
    "mhb_mercy_candidates_scratch_bytes", "mhb_mercy_candidates", "mhb_mercy_edges_scratch_bytes", "mhb_mercy_edges", "mhb_mercy_edges_count", "mhb_mercy_edges_write", "mhb_mercy_edges_segs", "mhb_mercy_host", "mhb_mercy_planes_words", "mhb_mercy_probe_owned", "mhb_mercy_count_planes", "mhb_edge_lut_bytes", "mhb_edge_lut_build",
    "mhb_release", "mhb_count_run", "mhb_count_run_multi", "mhb_seq2sdbg_run", "mhb_selftest_count_record", "mhb_selftest_count_records_roll", "mhb_selftest_s2s_record",
    "mhb_iterate_host", "mhb_iterate_run", "mhb_selftest_iterate", "mhb_s2s_extract_edges_pruned", "mhb_s2s_emit_fmt", "mhb_read2sdbg_host", "mhb_read2sdbg_run", "mhb_selftest_r2s_s1_record", "mhb_selftest_r2s_item",
    "mhb_selftest_kmsort", "mhb_selftest_kmsort_smem", "mhb_selftest_r2s_s1_group", "mhb_selftest_r2s_mercy_read",
]


def load():
    """Load libmhb.so; raises MhbError if it has not been built (python __graft_entry__.py / make)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MhbError(f"{LIB_PATH} is missing: build it with `make -C megahit_b200/csrc` "
                       "(there is no CPU fallback for the CUDA path)")
    L = C.CDLL(LIB_PATH)
    L.mhb_last_error.restype = C.c_char_p
    L.mhb_version.restype = C.c_char_p
    for f in ("mhb_count_record_words", "mhb_words_per_edge", "mhb_s2s_record_words", "mhb_count_sort_bytes",
              "mhb_s2s_sort_bytes"):
        getattr(L, f).restype = C.c_uint32
    for f in ("mhb_sort_workspace_bytes", "mhb_count_solid_scratch_bytes", "mhb_tipset_bytes",
              "mhb_s2s_emit_scratch_bytes"):
        getattr(L, f).restype = C.c_size_t
    L.mhb_sort_workspace_bytes.argtypes = [C.c_uint64, C.c_uint32]
    L.mhb_count_solid_scratch_bytes.argtypes = [C.c_uint64]
    L.mhb_tipset_bytes.argtypes = [C.c_uint64, C.c_uint32]
    L.mhb_s2s_emit_scratch_bytes.argtypes = [C.c_uint64, C.c_uint32]
    L.mhb_count_extract.argtypes = [C.c_void_p, C.POINTER(DevReads), C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p,
                                    C.c_int]
    L.mhb_sort_records.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32,
                                   C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]
    L.mhb_sort_records_relaxed.argtypes = L.mhb_sort_records.argtypes
    L.mhb_count_solid.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p,
                                  C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.mhb_count_hashed_workspace_bytes.restype = C.c_size_t
    L.mhb_count_hashed_workspace_bytes.argtypes = [C.c_uint64, C.c_uint32, C.c_int32]
    L.mhb_count_hashed_supported.argtypes = [C.c_uint32, C.c_int32]
    L.mhb_count_solid_hashed.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.mhb_tipset_build.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_size_t,
                                   C.c_uint64]
    L.mhb_count_mark_mercy.argtypes = [C.c_void_p, C.POINTER(DevReads), C.c_uint32, C.c_void_p, C.c_size_t, C.c_uint64,
                                       C.c_void_p, C.c_void_p]
    L.mhb_count_tip_edges.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.mhb_s2s_extract.argtypes = [C.c_void_p, C.POINTER(DevSeqs), C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p,
                                  C.c_int]
    L.mhb_s2s_emit.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_size_t]
    L.mhb_count_host.argtypes = [C.POINTER(CountArgs), C.POINTER(CountResult)]
    L.mhb_s2s_host.argtypes = [C.POINTER(S2sArgs), C.POINTER(S2sResult)]
    L.mhb_build_host.argtypes = [C.POINTER(BuildArgs), C.POINTER(BuildResult)]
    L.mhb_mercy_candidates_scratch_bytes.restype = C.c_size_t
    L.mhb_mercy_candidates_scratch_bytes.argtypes = [C.c_uint64]
    L.mhb_mercy_edges_scratch_bytes.restype = C.c_size_t
    L.mhb_mercy_edges_scratch_bytes.argtypes = [C.c_uint64, C.c_uint32]
    L.mhb_mercy_candidates.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64),
                                       C.c_void_p, C.c_size_t]
    L.mhb_mercy_edges.argtypes = [C.c_void_p, C.POINTER(DevReads), C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                  C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p,
                                  C.c_size_t]
    L.mhb_mercy_edges_segs.argtypes = [C.c_void_p, C.POINTER(DevReads), C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                       C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                       C.POINTER(C.c_uint64), C.c_void_p, C.c_size_t]
    L.mhb_mercy_edges_count.argtypes = [C.c_void_p, C.POINTER(DevReads), C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                        C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64),
                                        C.c_void_p, C.c_size_t]
    L.mhb_mercy_edges_write.argtypes = [C.c_void_p, C.POINTER(DevReads), C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                        C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_size_t]
    L.mhb_mercy_planes_words.restype = C.c_size_t
    L.mhb_mercy_planes_words.argtypes = [C.c_uint64, C.c_uint32]
    L.mhb_mercy_probe_owned.argtypes = [C.c_void_p, C.POINTER(DevReads), C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                        C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.mhb_mercy_count_planes.argtypes = [C.c_void_p, C.POINTER(DevReads), C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                         C.c_void_p, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p, C.c_size_t]
    L.mhb_plan_partition.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]
    L.mhb_edge_lut_bytes.restype = C.c_size_t
    L.mhb_edge_lut_build.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    L.mhb_sort_pass_ms.argtypes = [C.c_int, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64),
                                   C.POINTER(C.c_uint32)]
    L.mhb_set_device.argtypes = [C.c_int]
    L.mhb_partition_scatter.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_size_t]
    L.mhb_partition_scatter_hist.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    L.mhb_dev_malloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    L.mhb_dev_free.argtypes = [C.c_void_p]
    L.mhb_ipc_export.argtypes = [C.c_void_p, C.c_void_p]
    L.mhb_ipc_open.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.mhb_ipc_close.argtypes = [C.c_void_p]
    L.mhb_free.argtypes = [C.c_void_p]
    L.mhb_count_run.argtypes = [C.POINTER(CountOpts)]
    L.mhb_seq2sdbg_run.argtypes = [C.POINTER(Seq2SdbgOpts)]
    L.mhb_selftest_count_record.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                            C.POINTER(C.c_uint32)]
    L.mhb_selftest_count_records_roll.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                                  C.c_void_p]
    L.mhb_selftest_s2s_record.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                          C.c_uint32, C.c_void_p]
    L.mhb_s2s_emit_fmt.argtypes = L.mhb_s2s_emit.argtypes + [C.c_int]
    L.mhb_iterate_host.argtypes = [C.POINTER(IterateArgs), C.POINTER(IterateResult)]
    L.mhb_selftest_iterate.argtypes = [C.POINTER(IterateArgs), C.POINTER(IterateResult)]
    L.mhb_iterate_run.argtypes = [C.POINTER(IterateOpts)]
    L.mhb_s2s_extract_edges_pruned.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                               C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int]
    L.mhb_read2sdbg_host.argtypes = [C.POINTER(BuildArgs), C.POINTER(BuildResult)]
    L.mhb_read2sdbg_run.argtypes = [C.POINTER(Read2SdbgOpts)]
    L.mhb_selftest_r2s_s1_record.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p]
    L.mhb_selftest_r2s_item.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                        C.c_void_p, C.POINTER(C.c_uint32)]
    L.mhb_selftest_kmsort.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
    L.mhb_selftest_kmsort_smem.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
    L.mhb_selftest_r2s_s1_group.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_uint32, C.c_uint64, C.c_int,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mhb_selftest_r2s_mercy_read.argtypes = [C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        raise MhbError(f"libmhb error {rc}: {load().mhb_last_error().decode()}")


def device_count() -> int:
    return load().mhb_device_count()


def launch_count() -> int:
    """kernels launched through libmhb by this process so far"""
    L = load()
    L.mhb_launch_count.restype = C.c_uint64
    return int(L.mhb_launch_count())


# ------------------------------------------------------------------------------------------------
# geometry
# ------------------------------------------------------------------------------------------------
def plan_rounds(hist256, max_records: int):
    """Leading-byte ranges of the out-of-core count stage (host logic only): list of (lo, hi)."""
    L = load()
    h = np.ascontiguousarray(hist256, dtype=np.uint64)
    assert h.shape == (256,)
    lo, hi = (C.c_uint32 * 256)(), (C.c_uint32 * 256)()
    L.mhb_plan_rounds.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    n = L.mhb_plan_rounds(h.ctypes.data, int(max_records), lo, hi)
    if n < 0:
        raise MhbError(L.mhb_last_error().decode())
    return [(int(lo[i]), int(hi[i])) for i in range(n)]


def plan_rounds16(hist256, sub_hist, max_records: int, cap: int = 65536):
    """Two-level planner of the host rounds: list of (lo16, hi16) bucket-id ranges."""
    L = load()
    h = np.ascontiguousarray(hist256, dtype=np.uint64)
    sub = None if sub_hist is None else np.ascontiguousarray(sub_hist, dtype=np.uint64).reshape(256, 256)
    lo, hi = (C.c_uint32 * cap)(), (C.c_uint32 * cap)()
    L.mhb_plan_rounds16.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32]
    n = L.mhb_plan_rounds16(h.ctypes.data, sub.ctypes.data if sub is not None else None, int(max_records), lo, hi, cap)
    if n < 0:
        raise MhbError(L.mhb_last_error().decode())
    return [(int(lo[i]), int(hi[i])) for i in range(n)]


def set_round_limit(max_records: int = 0):
    """Cap the records per round of the out-of-core count stage (0 = derive from free device memory)."""
    L = load()
    L.mhb_set_round_limit.argtypes = [C.c_uint64]
    _check(L.mhb_set_round_limit(int(max_records)))


def set_s2s_round_limit(max_items: int = 0):
    """Cap the sort items per round of the out-of-core seq2sdbg stage (0 = derive from free device memory)."""
    L = load()
    L.mhb_set_s2s_round_limit.argtypes = [C.c_uint64]
    _check(L.mhb_set_s2s_round_limit(int(max_items)))


def mercy_host(k: int, edges: np.ndarray, cand_bin: np.ndarray) -> np.ndarray:
    """GenMercyEdges on the device from host buffers: sorted `.edges` records + the `.cand` image -> mercy edge records."""
    L = load()
    we = words_per_edge(k)
    edges = np.ascontiguousarray(edges, np.uint32).reshape(-1, we)
    cand = np.ascontiguousarray(cand_bin, np.uint32).reshape(-1)
    out, nm, nr = C.POINTER(C.c_uint32)(), C.c_uint64(), C.c_uint64()
    L.mhb_mercy_host.argtypes = [C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.POINTER(C.c_uint32)),
                                 C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    _check(L.mhb_mercy_host(k, edges.ctypes.data if len(edges) else None, len(edges), cand.ctypes.data if len(cand) else None,
                            len(cand), C.byref(out), C.byref(nm), C.byref(nr)))
    res = np.ctypeslib.as_array(out, (max(nm.value, 1) * we,))[: nm.value * we].reshape(-1, we).copy()
    L.mhb_free(out)
    return res


def sort_pass_ms(back: int = 0):
    """(per-pass ms list, n_records, words) of a recent sort; back=0 is the latest."""
    buf = (C.c_double * 80)()
    npass, nrec, words = C.c_uint32(), C.c_uint64(), C.c_uint32()
    _check(load().mhb_sort_pass_ms(back, buf, 80, C.byref(npass), C.byref(nrec), C.byref(words)))
    return list(buf[: npass.value]), nrec.value, words.value


def count_record_words(k: int) -> int:
    return load().mhb_count_record_words(C.c_uint32(k))


def words_per_edge(k: int) -> int:
    return load().mhb_words_per_edge(C.c_uint32(k))


def s2s_record_words(k: int) -> int:
    return load().mhb_s2s_record_words(C.c_uint32(k))


def count_sort_bytes(k: int) -> list[int]:
    buf = (C.c_uint8 * 80)()
    n = load().mhb_count_sort_bytes(C.c_uint32(k), buf)
    return list(buf[:n])


def s2s_sort_bytes(k: int) -> list[int]:
    buf = (C.c_uint8 * 80)()
    n = load().mhb_s2s_sort_bytes(C.c_uint32(k), buf)
    return list(buf[:n])


# ------------------------------------------------------------------------------------------------
# host level
# ------------------------------------------------------------------------------------------------
def count_host(bin_words: np.ndarray, n_reads: int, k: int, m: int, want_mercy: bool = True) -> dict:
    """KmerCounter::Run on host buffers.  bin_words: the `.bin` image as uint32 (numpy, or a pinned
    torch tensor's numpy view)."""
    L = load()
    bin_words = np.ascontiguousarray(bin_words, dtype=np.uint32).reshape(-1)
    a = CountArgs(k, m, bin_words.ctypes.data if len(bin_words) else None, len(bin_words), n_reads, int(want_mercy))
    r = CountResult()
    _check(L.mhb_count_host(C.byref(a), C.byref(r)))
    wpe = r.words_per_edge
    out = {
        "n_edge_records": r.n_edge_records, "n_solid": r.n_solid, "words_per_edge": wpe,
        "edges": np.ctypeslib.as_array(r.edges, (max(r.n_solid, 1) * wpe,))[: r.n_solid * wpe].reshape(-1, wpe).copy(),
        "cand_ids": (np.ctypeslib.as_array(r.cand_ids, (max(r.n_cand, 1),))[: r.n_cand].copy()
                     if want_mercy else np.zeros(0, np.uint64)),
        "n_has_tips": r.n_has_tips, "counting": np.array(r.counting, dtype=np.int64),
        "ms": {k_: getattr(r, f"t_{k_}_ms") for k_ in ("h2d", "extract", "sort", "count", "mercy", "d2h", "total")},
        "sort_pass_ms": list(r.sort_pass_ms[: r.n_sort_passes]), "n_rounds": int(r.n_rounds),
    }
    L.mhb_free(r.edges)
    if want_mercy:
        L.mhb_free(r.cand_ids)
    return out


def s2s_host(words: np.ndarray, word_off: np.ndarray, length: np.ndarray, mult: np.ndarray, k: int) -> dict:
    """SeqToSdbg::Run (after Initialize) on host buffers of package-orientation sequences."""
    L = load()
    words = np.ascontiguousarray(words, np.uint32)
    if len(words) == 0:
        words = np.zeros(1, np.uint32)
    word_off = np.ascontiguousarray(word_off, np.uint64)
    n = len(word_off) - 1
    length = np.ascontiguousarray(length, np.uint32) if n else np.zeros(1, np.uint32)
    mult = np.ascontiguousarray(mult, np.uint16) if n else np.zeros(1, np.uint16)
    a = S2sArgs(k, words.ctypes.data, word_off.ctypes.data, length.ctypes.data, mult.ctypes.data, n)
    r = S2sResult()
    _check(L.mhb_s2s_host(C.byref(a), C.byref(r)))
    table = np.array(r.bucket_table, np.uint64).reshape(NUM_BUCKETS, 4)
    out = {
        "n_records": r.n_records, "n_items": r.n_items, "n_tips": r.n_tips, "n_large_mul": r.n_large_mul,
        "n_bytes": r.n_bytes, "words_per_tip_label": r.words_per_tip_label,
        "bytes": bytes(np.ctypeslib.as_array(r.bytes, (max(r.n_bytes, 1),))[: r.n_bytes]),
        "bucket_table": table, "w_count": np.array(r.w_count, np.uint64), "ones_in_last": r.ones_in_last,
        "ms": {k_: getattr(r, f"t_{k_}_ms") for k_ in ("extract", "sort", "emit", "total")},
    }
    L.mhb_free(r.bytes)
    return out


def build_host(bin_words: np.ndarray, n_reads: int, k: int, m: int, need_mercy: bool = True, want_edges: bool = False,
               sdbg_out: np.ndarray | None = None, copy_bytes: bool = True) -> dict:
    """Fused k_min build: `.bin` image in, SdBG item stream out (count -> mercy edges -> seq2sdbg on the device).
    sdbg_out: optional (pinned) uint8 buffer that receives the stream."""
    L = load()
    bin_words = np.ascontiguousarray(bin_words, dtype=np.uint32).reshape(-1)
    a = BuildArgs(k, m, bin_words.ctypes.data if len(bin_words) else None, len(bin_words), n_reads, int(need_mercy),
                  int(want_edges), sdbg_out.ctypes.data if sdbg_out is not None else None,
                  sdbg_out.nbytes if sdbg_out is not None else 0)
    r = BuildResult()
    _check(L.mhb_build_host(C.byref(a), C.byref(r)))
    in_place = sdbg_out is not None and C.addressof(r.bytes.contents) == sdbg_out.ctypes.data if r.n_bytes else sdbg_out is not None
    out = {
        "n_edge_records": r.n_edge_records, "n_solid": r.n_solid, "n_cand": r.n_cand, "n_mercy": r.n_mercy,
        "n_sort_items": r.n_sort_items, "n_items": r.n_items, "n_tips": r.n_tips, "n_large_mul": r.n_large_mul,
        "n_bytes": r.n_bytes, "words_per_tip_label": r.words_per_tip_label,
        "bucket_table": np.ctypeslib.as_array(r.bucket_table, (NUM_BUCKETS * 4,)).reshape(NUM_BUCKETS, 4).copy(),
        "w_count": np.array(r.w_count, np.uint64), "ones_in_last": r.ones_in_last,
        "ms": {k_: getattr(r, f"t_{k_}_ms") for k_ in ("total", "h2d", "count", "mercy", "s2s", "d2h")},
    }
    if copy_bytes:
        out["bytes"] = bytes(np.ctypeslib.as_array(r.bytes, (max(r.n_bytes, 1),))[: r.n_bytes])
    if not in_place:
        L.mhb_free(r.bytes)
    L.mhb_free(r.bucket_table)
    if want_edges:
        wpe = r.words_per_edge
        out["edges"] = np.ctypeslib.as_array(r.edges, (max(r.n_solid, 1) * wpe,))[: r.n_solid * wpe].reshape(-1, wpe).copy()
        out["cand_ids"] = np.ctypeslib.as_array(r.cand_ids, (max(r.n_cand, 1),))[: r.n_cand].copy()
        out["counting"] = np.ctypeslib.as_array(r.counting, (65536,)).copy()
        L.mhb_free(r.edges)
        L.mhb_free(r.cand_ids)
        L.mhb_free(r.counting)
    return out


def read2sdbg_host(bin_words: np.ndarray, n_reads: int, k: int, m: int, need_mercy: bool = True) -> dict:
    """The 1-pass build (`megahit_core read2sdbg`, main_sdbg_build.cpp:88-156): `.bin` image in, SdBG item stream out,
    plus what stage 1 writes to P.counting."""
    L = load()
    bin_words = np.ascontiguousarray(bin_words, dtype=np.uint32).reshape(-1)
    a = BuildArgs(k, m, bin_words.ctypes.data if len(bin_words) else None, len(bin_words), n_reads, int(need_mercy), 0, None, 0)
    r = BuildResult()
    _check(L.mhb_read2sdbg_host(C.byref(a), C.byref(r)))
    out = {
        "n_edge_records": r.n_edge_records, "n_distinct_items": r.n_solid, "n_mercy": r.n_mercy,
        "n_sort_items": r.n_sort_items, "n_items": r.n_items, "n_tips": r.n_tips, "n_large_mul": r.n_large_mul,
        "n_bytes": r.n_bytes, "words_per_tip_label": r.words_per_tip_label,
        "bucket_table": np.ctypeslib.as_array(r.bucket_table, (NUM_BUCKETS * 4,)).reshape(NUM_BUCKETS, 4).copy(),
        "w_count": np.array(r.w_count, np.uint64), "ones_in_last": r.ones_in_last,
        "counting": np.ctypeslib.as_array(r.counting, (65536,)).copy(),
        "bytes": bytes(np.ctypeslib.as_array(r.bytes, (max(r.n_bytes, 1),))[: r.n_bytes]),
        "ms": {"total": r.t_total_ms, "h2d": r.t_h2d_ms, "s1_records_partition": r.t_count_ms, "kmsort": r.t_mercy_ms,
               "stage2": r.t_s2s_ms, "d2h": r.t_d2h_ms},
    }
    L.mhb_free(r.bytes)
    L.mhb_free(r.bucket_table)
    L.mhb_free(r.counting)
    return out


def sdbg_stream_from_table(table: np.ndarray, data: bytes) -> bytes:
    """Canonical SdBG stream (formats.canonical_sdbg) from the {offset, items, tips, large} table."""
    chunks = []
    wpt_unknown = None  # byte extents follow from the next non-empty bucket's offset
    idx = np.nonzero(table[:, 1])[0]
    ends = list(table[idx[1:], 0]) + [len(data)] if len(idx) else []
    for b, end in zip(idx, ends):
        chunks.append(np.array([b], "<u4").tobytes() + np.array([table[b, 1]], "<u8").tobytes()
                      + data[int(table[b, 0]):int(end)])
    del wpt_unknown
    return b"".join(chunks)


# ------------------------------------------------------------------------------------------------
# file level (the sub-commands)
# ------------------------------------------------------------------------------------------------
def count_run(read_lib_file: str, output_prefix: str, k: int = 21, m: int = 2, host_mem: float = 1e9,
              num_cpu_threads: int = 0, mem_flag: int = 1) -> None:
    o = CountOpts(k, m, host_mem, num_cpu_threads, read_lib_file.encode(), output_prefix.encode(), mem_flag)
    _check(load().mhb_count_run(C.byref(o)))


def seq2sdbg_run(output_prefix: str, k: int, k_from: int = 0, input_prefix: str = "", contig: str = "",
                 bubble: str = "", addi_contig: str = "", local_contig: str = "", need_mercy: bool = False,
                 host_mem: float = 1e9, num_cpu_threads: int = 0, mem_flag: int = 1) -> None:
    o = Seq2SdbgOpts(host_mem, k, k_from, num_cpu_threads, contig.encode(), bubble.encode(), addi_contig.encode(),
                     local_contig.encode(), input_prefix.encode(), output_prefix.encode(), int(need_mercy), mem_flag)
    _check(load().mhb_seq2sdbg_run(C.byref(o)))


def iterate_host(contig_words: np.ndarray, contig_word_off: np.ndarray, contig_len: np.ndarray, bin_words: np.ndarray,
                 n_reads: int, k: int, step: int, selftest: bool = False) -> dict:
    """`megahit_core iterate` (main_iterate.cpp): contigs (file orientation, flag-filtered) + read library in, the set of
    iterative edges for k + step out (ascending `.edges` records, multiplicity 0).  selftest: the host mirror of the
    device code (CPU tests), not a compute path."""
    L = load()
    cw = np.ascontiguousarray(contig_words, np.uint32)
    if len(cw) == 0:
        cw = np.zeros(1, np.uint32)
    co = np.ascontiguousarray(contig_word_off, np.uint64)
    cl = np.ascontiguousarray(contig_len, np.uint32)
    n_contigs = len(cl)
    if n_contigs == 0:
        cl = np.zeros(1, np.uint32)
    b = np.ascontiguousarray(bin_words, np.uint32).reshape(-1)
    a = IterateArgs(k, step, cw.ctypes.data, co.ctypes.data, cl.ctypes.data, n_contigs, b.ctypes.data if len(b) else None,
                    len(b), n_reads)
    r = IterateResult()
    _check((L.mhb_selftest_iterate if selftest else L.mhb_iterate_host)(C.byref(a), C.byref(r)))
    W = r.words_per_edge
    out = {"n_flanks": r.n_flanks, "n_aligned_reads": r.n_aligned_reads, "n_candidates": r.n_candidates, "n_edges": r.n_edges,
           "edges": np.ctypeslib.as_array(r.edges, (max(r.n_edges, 1) * W,))[: r.n_edges * W].reshape(-1, W).copy(),
           "ms": r.t_total_ms}
    L.mhb_free(r.edges)
    return out


def iterate_run(contig_file: str, bubble_file: str, read_file: str, output_prefix: str, k: int, step: int,
                num_cpu_threads: int = 0) -> None:
    o = IterateOpts(contig_file.encode(), bubble_file.encode(), read_file.encode(), num_cpu_threads, k, step,
                    output_prefix.encode())
    _check(load().mhb_iterate_run(C.byref(o)))


def read2sdbg_run(read_lib_file: str, output_prefix: str, k: int = 21, m: int = 2, need_mercy: bool = False,
                  host_mem: float = 1e9, num_cpu_threads: int = 0, mem_flag: int = 1) -> None:
    o = Read2SdbgOpts(k, m, host_mem, num_cpu_threads, read_lib_file.encode(), output_prefix.encode(), mem_flag,
                      int(need_mercy))
    _check(load().mhb_read2sdbg_run(C.byref(o)))


# ------------------------------------------------------------------------------------------------
# self-test hooks (host, one record at a time)
# ------------------------------------------------------------------------------------------------
def selftest_count_record(read_words: np.ndarray, L_: int, k: int, q: int):
    read_words = np.ascontiguousarray(read_words, np.uint32)
    rec = np.zeros(count_record_words(k), np.uint32)
    strand = C.c_uint32()
    _check(load().mhb_selftest_count_record(read_words.ctypes.data, len(read_words), L_, k, q, rec.ctypes.data,
                                            C.byref(strand)))
    return rec, strand.value


def selftest_count_records_roll(read_words: np.ndarray, L_: int, k: int, q: int):
    """4 consecutive 8-byte count records from position q on, built by the rolling builder (host run)."""
    read_words = np.ascontiguousarray(read_words, np.uint32)
    rec = np.zeros(4, np.uint64)
    strand = np.zeros(4, np.uint32)
    _check(load().mhb_selftest_count_records_roll(read_words.ctypes.data, len(read_words), L_, k, q, rec.ctypes.data,
                                                  strand.ctypes.data))
    return rec, strand


def selftest_s2s_record(seq_words: np.ndarray, L_: int, k: int, strand: int, offset: int, mult: int):
    seq_words = np.ascontiguousarray(seq_words, np.uint32)
    rec = np.zeros(s2s_record_words(k), np.uint32)
    _check(load().mhb_selftest_s2s_record(seq_words.ctypes.data, len(seq_words), L_, k, strand, offset, mult,
                                          rec.ctypes.data))
    return rec


def r2s_s1_key_words(k: int) -> int:
    return (2 * (k - 1) + 6 + 31) // 32


def selftest_r2s_s1_record(pkg_words: np.ndarray, L_: int, k: int, e: int, base_off: int = 0):
    """stage-1 record number e (bucket input order) of a package-orientation read: key words + 2 payload words"""
    pkg_words = np.ascontiguousarray(pkg_words, np.uint32)
    rec = np.zeros(r2s_s1_key_words(k) + 2, np.uint32)
    _check(load().mhb_selftest_r2s_s1_record(pkg_words.ctypes.data, len(pkg_words), L_, k, e, base_off, rec.ctypes.data))
    return rec


def selftest_r2s_item(pkg_words: np.ndarray, L_: int, k: int, i: int, strand: int, type_: int):
    pkg_words = np.ascontiguousarray(pkg_words, np.uint32)
    rec = np.zeros(s2s_record_words(k), np.uint32)
    pal = C.c_uint32()
    _check(load().mhb_selftest_r2s_item(pkg_words.ctypes.data, len(pkg_words), L_, k, i, strand, type_, rec.ctypes.data,
                                        C.byref(pal)))
    return rec, pal.value


def selftest_kmsort(recs: np.ndarray, nw: int, smem: bool = False, cap: int = 65535, wcap: int = 0) -> np.ndarray:
    """kmlib::kmsort's permutation of one bucket (records of nw + 2 words), emulated level by level as on the device:
    the in-place walk on the records, or (smem) the walk on tags + staged ranges the default kernels use"""
    recs = np.ascontiguousarray(recs, np.uint32).copy()
    if smem:
        _check(load().mhb_selftest_kmsort_smem(recs.ctypes.data, len(recs), nw, cap, wcap))
    else:
        _check(load().mhb_selftest_kmsort(recs.ctypes.data, len(recs), nw))
    return recs
