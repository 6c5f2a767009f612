"""Multi-GPU SdBG build: one process per GPU, `torch.distributed` (NCCL over NVLink/NVSwitch) for the exchange.

The path shards naturally (SURVEY.md 8e): both stages are "extract locally -> all records with the same
leading bases must meet -> sort + scan locally -> own a contiguous range of the 65 536 prefix buckets".
The reference already treats prefix buckets as independent (sorting/base_engine.cpp:323-326) and both
on-disk formats map bucket -> (file, offset), so every rank can write its own `.edges.<r>` / `.sdbg.<r>`
with no merge.

Partition key = the record's most significant byte (its first 4 bases), cut into `world` CONTIGUOUS
ranges chosen from the all-reduced 256-bin histogram so that every rank receives about the same number of
records (canonical (k+1)-mers are skewed towards A-prefixes, equal-width ranges would not balance).  A
contiguous range of the top byte is a contiguous range of bucket ids, which is what `.edges.info` /
`.sdbg_info` can express - a whole-edge minimizer hash could not (SURVEY.md 8e).

Per stage and rank:   extract (+ histogram of the top byte)  ->  one stable radix pass on the top byte
(groups records by destination)  ->  ONE variable-size all-to-all  ->  LSD radix sort of the received
records  ->  count / emit for the owned buckets.  Cross-rank state besides the two record exchanges:
the 256-bin histograms (all-reduce), the tip edges (all-gather, tiny) for the per-read mercy marks, and
the solid edges (all-gather) for the mercy-edge searches.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch
import torch.distributed as dist

from . import lib
from .dev import _ptr, _stream, sort_records


def plan_ranges(hist: np.ndarray, world: int) -> np.ndarray:
    """Cut the 256 top-byte values into `world` contiguous, non-empty ranges with near-equal record counts.
    Returns bounds[world+1] (bounds[0] = 0, bounds[world] = 256); rank r owns [bounds[r], bounds[r+1])."""
    assert 1 <= world <= 256
    cum = np.concatenate([[0], np.cumsum(np.asarray(hist).astype(np.int64))])
    total = int(cum[-1])
    bounds = [0]
    for r in range(1, world):
        lo, hi = bounds[-1] + 1, 256 - (world - r)  # leave at least one value for every later rank
        target = total * r // world
        cand = np.arange(lo, hi + 1)
        bounds.append(int(cand[np.argmin(np.abs(cum[cand] - target))]))
    bounds.append(256)
    return np.array(bounds, np.int64)


def split_counts(hist: np.ndarray, bounds: np.ndarray) -> np.ndarray:
    cum = np.concatenate([[0], np.cumsum(hist.astype(np.int64))])
    return (cum[bounds[1:]] - cum[bounds[:-1]]).astype(np.int64)


def exchange_records(grouped: torch.Tensor, words: int, send_counts: np.ndarray, group=None) -> torch.Tensor:
    """grouped: int32 tensor of records already grouped by destination rank (ascending); returns the
    records this rank owns (concatenated in source-rank order)."""
    world = dist.get_world_size(group)
    sc = torch.tensor(send_counts, dtype=torch.int64, device=grouped.device)
    rc = torch.empty_like(sc)
    dist.all_to_all_single(rc, sc, group=group)
    recv_counts = rc.cpu().numpy()
    n_recv = int(recv_counts.sum())
    out = torch.empty(n_recv * words + 4, dtype=torch.int32, device=grouped.device)
    n_send = int(send_counts.sum())
    dist.all_to_all_single(out[: n_recv * words], grouped[: n_send * words],
                           output_split_sizes=[int(c) * words for c in recv_counts],
                           input_split_sizes=[int(c) * words for c in send_counts], group=group)
    assert world == len(send_counts)
    return out, n_recv


class _RawView:
    """int32 torch view over raw (cudaMalloc'ed) device memory, via the CUDA array interface"""

    def __init__(self, ptr, nelem):
        self.__cuda_array_interface__ = {"shape": (int(nelem),), "typestr": "<i4", "data": (int(ptr), False), "version": 3}


class PeerBuffers:
    """One receive buffer per rank for a stage, cudaMalloc'ed by libmhb and opened on every rank through CUDA IPC,
    so that a rank's partition kernel can store records straight into their owner's memory over NVLink."""

    def __init__(self, nbytes: int):
        L = lib.load()
        self.L, self.nbytes = L, int(nbytes)
        p = C.c_void_p()
        lib._check(L.mhb_dev_malloc(C.byref(p), self.nbytes))
        self.ptr = p.value
        h = (C.c_uint8 * 64)()
        lib._check(L.mhb_ipc_export(C.c_void_p(self.ptr), h))
        handles = [None] * dist.get_world_size()
        dist.all_gather_object(handles, bytes(h))
        self.peers = []
        for r, hb in enumerate(handles):
            if r == dist.get_rank():
                self.peers.append(self.ptr)
            else:
                q = C.c_void_p()
                buf = (C.c_uint8 * 64).from_buffer_copy(hb)
                lib._check(L.mhb_ipc_open(buf, C.byref(q)))
                self.peers.append(q.value)
        self.peers_c = (C.c_uint64 * 16)(*self.peers)
        dist.barrier()

    def close(self):
        dist.barrier()
        for r, q in enumerate(self.peers):
            if r != dist.get_rank():
                self.L.mhb_ipc_close(C.c_void_p(q))
        dist.barrier()
        self.L.mhb_dev_free(C.c_void_p(self.ptr))


class MultiGpuBuild:
    """count -> mercy -> seq2sdbg across the ranks of the default process group (fixed-length reads).

    Host involvement per step is limited to reading a handful of counters (records owned, solid edges, tips,
    candidates, mercy edges) that size the next launches; plans, owner tables and destination addresses are computed
    on the device (mhb_plan_partition) from one all-gather of the 256-bin histograms, and the ranks order their
    accesses to each other's buffers with stream-ordered collectives (the histogram all-gather before the scatter, a
    one-word all-reduce after it) instead of host barriers."""

    def __init__(self, n_reads: int, read_len: int, k: int, m: int, device, need_mercy: bool = True):
        import os
        self.L = lib.load()
        self.n_reads, self.read_len, self.k, self.m, self.device = n_reads, read_len, k, m, device
        self.need_mercy = need_mercy
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        if self.world > 16:
            raise lib.MhbError("the multi-GPU build supports up to 16 ranks (one node)")
        self.WR, self.WE, self.W2 = lib.count_record_words(k), lib.words_per_edge(k), lib.s2s_record_words(k)
        self.cbytes, self.sbytes = lib.count_sort_bytes(k), lib.s2s_sort_bytes(k)
        self.n_local = n_reads * (read_len - k) if read_len >= k + 1 else 0
        self.stride = 1 + (read_len + 15) // 16
        self.times = {}
        self.fused = self.world > 1 and not os.environ.get("MHB_MGPU_NCCL_A2A")
        # count stage on the owned records: two partition passes + per-bucket hash aggregation where available
        self.hashed = bool(self.L.mhb_count_hashed_supported(k, m)) and os.environ.get("MHB_COUNT_MODE", "auto") != "sort"
        self.peer = {}
        self._bufs = {}
        self._tok = torch.zeros(1, dtype=torch.int32, device=device)
        self._pin = torch.empty(64, dtype=torch.int64).pin_memory()
        self._timed = False

    # ------------------------------------------------------------------ helpers
    def _mark(self, name):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        self.times.setdefault(name, []).append(ev)

    def _buf(self, name, numel, dtype=torch.int32, slack=1.0):
        """grow-only named device buffer: steady-state steps allocate nothing"""
        t = self._bufs.get(name)
        if t is None or t.numel() < numel or t.dtype != dtype:
            t = torch.empty(int(numel * slack) + 64, dtype=dtype, device=self.device)
            self._bufs[name] = t
        return t

    def _to_host(self, t: torch.Tensor) -> np.ndarray:
        """small device int64 tensor -> numpy through one pinned staging buffer (ONE stream sync)"""
        n = t.numel()
        self._pin[:n].copy_(t.reshape(-1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._pin[:n].numpy().copy()

    def _stream_barrier(self):
        """every rank's earlier work on its stream is complete before any rank's later work starts (no host sync)"""
        dist.all_reduce(self._tok)

    def _gather_counts(self, *vals) -> np.ndarray:
        """all-gather a few host integers; returns an array [world][len(vals)] (one sync)"""
        t = torch.tensor(list(vals), dtype=torch.int64, device=self.device)
        out = torch.empty(self.world * len(vals), dtype=torch.int64, device=self.device)
        dist.all_gather_into_tensor(out, t)
        return self._to_host(out).reshape(self.world, len(vals))

    def _peer(self, tag, need_bytes):
        """(re)allocate the IPC receive buffers of a stage - a collective: `need_bytes` must be the same on every rank"""
        pb = self.peer.get(tag)
        if pb is not None:
            pb.close()
        pb = self.peer[tag] = PeerBuffers(int(need_bytes * 1.25) + 4096)
        return pb

    def _partition_and_exchange(self, recs, n, words, top_byte, hist_dev, tag, expect_own, next_byte=None):
        """Move every record to the rank owning its leading byte.  Fused mode: ONE kernel does partition + exchange -
        the radix pass's scatter stores go straight into the owners' receive buffers over NVLink (CUDA IPC peer
        pointers).  Fallback (MHB_MGPU_NCCL_A2A=1): local pass, then one variable-size NCCL all-to-all.
        next_byte: the byte the owner's sort visits first - the fused exchange pass also counts that byte per owner, the
        ranks swap the 256-bin rows, and self._first_hist (device int64[256]; None on the fallback path or without
        next_byte) is the first-pass histogram of the owned records: the owner's sort need not sweep them to count.
        Returns (pointer to the owned records, count, bounds[world+1] numpy, owner table numpy uint8[256])."""
        L, W = self.L, self.world
        rb = words * 4
        self._first_hist = None
        hist_all = self._buf(tag + "_hist_all", W * 256, torch.int64)
        # the all-gather also orders the ranks: when it completes, every rank has finished the previous step's reads
        # of its receive buffer, so the scatter below may overwrite it
        dist.all_gather_into_tensor(hist_all[: W * 256], hist_dev)
        lut_dev = self._buf(tag + "_lut", 256, torch.uint8)
        addr_dev = self._buf(tag + "_addr", 256, torch.int64)
        plan_dev = self._buf(tag + "_plan", 64, torch.int64)
        # the receive buffers have the SAME size on every rank, derived from the plan (identical everywhere), so that all
        # ranks take the same (collective) reallocation decision; expect_own only matters for the log
        pb = self.peer.get(tag) if self.fused else None
        for attempt in range(2):
            peers_c = pb.peers_c if pb is not None else (C.c_uint64 * 16)()
            lib._check(L.mhb_plan_partition(_stream(), _ptr(hist_all), W, self.rank, rb, peers_c, _ptr(lut_dev), _ptr(addr_dev),
                                            _ptr(plan_dev)))
            plan = self._to_host(plan_dev[:64])
            recv_tot, send, bounds = plan[:W], plan[16:16 + W], plan[32:33 + W]
            self._recv_tot = recv_tot
            need = int(recv_tot.max()) * rb + 64
            if not self.fused or (pb is not None and need <= pb.nbytes):
                break
            pb = self._peer(tag, need)  # addresses change: plan once more
        owner = np.repeat(np.arange(W, dtype=np.uint8), np.diff(bounds).astype(np.int64))
        if self._timed:
            self._mark(tag + "_plan")
        ws = self._buf(tag + "_ws", L.mhb_sort_workspace_bytes(max(n, 1), words), torch.uint8)
        n_own = int(recv_tot[self.rank])
        if not self.fused:
            tmp = self._buf(tag + "_part", recs.numel())
            grouped = sort_records(recs, tmp, n, words, [top_byte], hist_dev, ws)
            sc = torch.tensor(send, dtype=torch.int64, device=recs.device)
            rc = torch.empty_like(sc)
            dist.all_to_all_single(rc, sc)
            recv_counts = self._to_host(rc)
            out = self._buf(tag + "_own", n_own * words + 4, slack=1.15)
            dist.all_to_all_single(out[: n_own * words], grouped[: int(send.sum()) * words],
                                   output_split_sizes=[int(c) * words for c in recv_counts],
                                   input_split_sizes=[int(c) * words for c in send])
            return out.data_ptr(), n_own, bounds, owner
        self._first_hist = None
        if next_byte is None:
            lib._check(L.mhb_partition_scatter(_stream(), _ptr(recs), n, words, top_byte, _ptr(lut_dev), _ptr(addr_dev), _ptr(ws),
                                               ws.numel()))
            self._stream_barrier()  # all ranks' scatter kernels have completed: my buffer is complete
            return pb.ptr, n_own, bounds, owner
        oh = self._buf(tag + "_ohist", 16 * 256, torch.int64)[: 16 * 256]
        oh.zero_()
        done = C.c_int(0)
        lib._check(L.mhb_partition_scatter_hist(_stream(), _ptr(recs), n, words, top_byte, _ptr(lut_dev), _ptr(addr_dev), _ptr(ws),
                                                ws.numel(), next_byte, _ptr(oh), C.byref(done)))
        # row o of my table goes to rank o; the all-to-all is also the barrier after the scatter
        got = self._buf(tag + "_ohist_in", W * 256, torch.int64)[: W * 256]
        dist.all_to_all_single(got, oh[: W * 256])
        self._first_hist = got.view(W, 256).sum(0).contiguous()
        return pb.ptr, n_own, bounds, owner

    def close(self):
        for pb in self.peer.values():
            pb.close()
        self.peer = {}

    def _sort_raw(self, ptr_a, n, words, sort_bytes, tag, first_hist=None):
        """LSD sort of n records at raw device pointer ptr_a; returns the pointer holding the result."""
        L = self.L
        tmp = self._buf(tag + "_tmp", n * words + 4, slack=1.15)
        ws = self._buf(tag + "_ws2", L.mhb_sort_workspace_bytes(max(n, 1), words), torch.uint8)
        arr = (C.c_uint8 * len(sort_bytes))(*sort_bytes)
        in_b = C.c_int(0)
        lib._check(L.mhb_sort_records_relaxed(_stream(), C.c_void_p(ptr_a), _ptr(tmp), n, words, arr, len(sort_bytes),
                                              _ptr(first_hist), _ptr(ws), ws.numel(), C.byref(in_b)))
        return tmp.data_ptr() if in_b.value else ptr_a

    # ------------------------------------------------------------------ mercy stage
    def _mercy(self, reads, bin_dev, edges, aux, n_solid, n_tip, owner):
        """tip edges of every rank -> per-read marks -> candidate reads -> searches answered by the owners of the
        searched prefixes -> mercy edges appended behind this rank's solid edges.  Returns (edges tensor, n_cand, n_mercy)."""
        L, k, dev, W, WE = self.L, self.k, self.device, self.world, self.WE
        i32 = dict(dtype=torch.int32, device=dev)
        e2 = edges[: n_solid * WE].view(-1, WE)
        # ---- tip edges of all ranks (0.5 % of the solid edges): one padded all-gather, padding has aux = 0 ----
        cnt = self._gather_counts(n_tip, n_solid)
        mx = max(int(cnt[:, 0].max()), 1)
        pad_t = self._buf("tip_pad", mx * WE)[: mx * WE].view(mx, WE)
        pad_a = self._buf("tip_pad_a", mx, torch.uint8)[:mx]
        pad_a.zero_()
        if n_tip:
            idx = torch.nonzero(aux[:n_solid]).reshape(-1)
            pad_t[:n_tip] = e2[idx]
            pad_a[:n_tip] = aux[:n_solid][idx]
        all_t = self._buf("tip_all", W * mx * WE)[: W * mx * WE]
        all_a = self._buf("tip_all_a", W * mx, torch.uint8)[: W * mx]
        dist.all_gather_into_tensor(all_t, pad_t.reshape(-1))
        dist.all_gather_into_tensor(all_a, pad_a)
        n_tip_all = int(cnt[:, 0].sum())
        need = L.mhb_tipset_bytes(n_tip_all, k)
        tipset = self._buf("tipset", need, torch.uint8, slack=1.2)
        lib._check(L.mhb_tipset_build(_stream(), _ptr(all_t), _ptr(all_a), W * mx, k, _ptr(tipset), need, n_tip_all))
        first = self._buf("first", self.n_reads + 1)
        last = self._buf("last", self.n_reads + 1)
        lib._check(L.mhb_count_mark_mercy(_stream(), C.byref(reads), k, _ptr(tipset), need, n_tip_all, _ptr(first), _ptr(last)))
        cand = self._buf("cand", self.n_reads + 1, torch.int64)
        cs = self._buf("cand_scratch", L.mhb_mercy_candidates_scratch_bytes(self.n_reads), torch.uint8)
        nc = C.c_uint64(0)
        lib._check(L.mhb_mercy_candidates(_stream(), _ptr(first), _ptr(last), self.n_reads, _ptr(cand), C.byref(nc), _ptr(cs),
                                          cs.numel()))
        n_cand = nc.value
        # ---- candidate reads of all ranks, padded (a zero length word = no positions) ----
        ccnt = self._gather_counts(n_cand)[:, 0]
        mc = int(ccnt.max())
        if mc == 0:
            return edges, 0, 0
        st = self.stride
        cpad = self._buf("cand_pad", mc * st)[: mc * st].view(mc, st)
        cpad.zero_()
        if n_cand:
            cpad[:n_cand] = bin_dev[: self.n_reads * st].view(self.n_reads, st)[cand[:n_cand]]
        call = self._buf("cand_all", W * mc * st + 8)
        dist.all_gather_into_tensor(call[: W * mc * st], cpad.reshape(-1))
        # ---- every rank answers the searches that land in its own bucket range, for ALL candidates ----
        lut = self._buf("edge_lut", L.mhb_edge_lut_bytes(), torch.uint8)
        lib._check(L.mhb_edge_lut_build(_stream(), _ptr(edges), n_solid, k, _ptr(lut)))
        pw = L.mhb_mercy_planes_words(mc, self.read_len)  # per source rank
        planes = self._buf("planes", W * pw)
        greads = lib.DevReads(call.data_ptr(), W * mc * st, W * mc, self.read_len, None, None)
        owner_c = (C.c_uint8 * 256)(*owner.tolist())
        lib._check(L.mhb_mercy_probe_owned(_stream(), C.byref(greads), None, W * mc, self.read_len, k, _ptr(edges), n_solid,
                                           _ptr(lut), owner_c, self.rank, _ptr(planes)))
        # planes[o] = my answers about rank o's candidates  ->  mine[s] = rank s's answers about MY candidates
        mine = self._buf("planes_mine", W * pw)
        dist.all_to_all_single(mine[: W * pw], planes[: W * pw])
        n_mercy = 0
        if n_cand:
            ms = self._buf("mercy_scratch", L.mhb_mercy_edges_scratch_bytes(n_cand, self.read_len) - L.mhb_edge_lut_bytes(),
                           torch.uint8, slack=1.2)
            nm = C.c_uint64(0)
            lib._check(L.mhb_mercy_count_planes(_stream(), C.byref(reads), _ptr(cand), n_cand, self.read_len, k, _ptr(mine), W, pw,
                                                C.byref(nm), _ptr(ms), ms.numel()))
            n_mercy = nm.value
            if n_mercy:
                have = edges.numel() // WE
                if n_solid + n_mercy > have:  # reads overlapping only at their ends: more mercy than solid edges
                    big = self._buf("edges_big", (n_solid + n_mercy) * WE + 4, slack=1.1)
                    big[: n_solid * WE].copy_(edges[: n_solid * WE])
                    edges = big
                lib._check(L.mhb_mercy_edges_write(_stream(), C.byref(reads), _ptr(cand), n_cand, self.read_len, k,
                                                   C.c_void_p(edges.data_ptr() + n_solid * WE * 4), n_mercy, n_mercy, _ptr(ms),
                                                   ms.numel()))
        return edges, n_cand, n_mercy

    # ------------------------------------------------------------------ one step
    def run(self, bin_dev: torch.Tensor, timed: bool = False) -> dict:
        L, k, m, dev = self.L, self.k, self.m, self.device
        self._timed = timed
        reads = lib.DevReads(bin_dev.data_ptr(), bin_dev.numel(), self.n_reads, self.read_len, None, None)
        if timed:
            self._mark("t0")
        # ---- count stage ----
        n = self.n_local
        a = self._buf("c_a", n * self.WR + 4)
        hist = self._buf("c_hist", 256, torch.int64)[:256]
        hist.zero_()
        top = self.cbytes[-1]
        lib._check(L.mhb_count_extract(_stream(), C.byref(reads), k, _ptr(a), n, _ptr(hist), top))
        if timed:
            self._mark("extract")
        c_first = 5 if self.hashed else self.cbytes[0]  # the byte the owner's count stage sorts on first
        own, n_own, bounds, owner = self._partition_and_exchange(a, n, self.WR, top, hist, "c", max(n, 1), next_byte=c_first)
        c_hist = self._first_hist
        if timed:
            self._mark("exchange1")
        cap = n_own // max(1, m) + 1
        edges = self._buf("edges", cap * self.WE + 4, slack=1.15)
        aux = self._buf("aux", cap, torch.uint8, slack=1.15)
        mul_hist = self._buf("mul_hist", 65536, torch.int64)[:65536]
        mul_hist.zero_()
        nsol = self._buf("nsol", 8, torch.int64)[:8]
        nsol.zero_()
        if self.hashed:
            if timed:
                self._mark("sort1")  # the two partition passes run inside the hashed count call
            tmp = self._buf("c_tmp", n_own * self.WR + 4, slack=1.15)
            hws = self._buf("c_hws", L.mhb_count_hashed_workspace_bytes(max(n_own, 1), k, m), torch.uint8, slack=1.15)
            lib._check(L.mhb_count_solid_hashed(_stream(), C.c_void_p(own), _ptr(tmp), n_own, k, m, _ptr(c_hist), _ptr(edges), _ptr(aux),
                                                cap, _ptr(mul_hist), _ptr(nsol), _ptr(hws), hws.numel()))
        else:
            srt = self._sort_raw(own, n_own, self.WR, self.cbytes, "c", c_hist)
            if timed:
                self._mark("sort1")
            scratch = self._buf("c_scratch", L.mhb_count_solid_scratch_bytes(n_own), torch.uint8, slack=1.15)
            lib._check(L.mhb_count_solid(_stream(), C.c_void_p(srt), n_own, k, m, _ptr(edges), _ptr(aux), cap, _ptr(mul_hist),
                                         _ptr(nsol), _ptr(scratch), scratch.numel()))
        dist.all_reduce(mul_hist)  # edge_counter.h:44-52: `.counting` is a global histogram
        n_solid = int(self._to_host(nsol[:1])[0])
        if n_solid > cap:
            raise lib.MhbError("internal: solid edges exceed capacity")
        n_tip = int((aux[:n_solid] != 0).sum().item()) if (self.need_mercy and n_solid) else 0
        if timed:
            self._mark("count")

        # ---- mercy ----
        n_mercy = n_cand = 0
        seq_edges = edges
        if self.need_mercy:
            seq_edges, n_cand, n_mercy = self._mercy(reads, bin_dev, edges, aux, n_solid, n_tip, owner)
        if timed:
            self._mark("mercy")

        # ---- seq2sdbg stage ----
        n_seqs = n_solid + n_mercy
        n_items = n_seqs * 6
        seqs = lib.DevSeqs(seq_edges.data_ptr(), n_seqs * self.WE, n_seqs, k + 1, None, None, None, None, self.WE)
        sa = self._buf("s_a", n_items * self.W2 + 4, slack=1.1)
        hist2 = self._buf("s_hist", 256, torch.int64)[:256]
        hist2.zero_()
        top2 = self.sbytes[-1]
        if os.environ.get("MHB_S2S_NO_PRUNE"):
            lib._check(L.mhb_s2s_extract(_stream(), C.byref(seqs), k, _ptr(sa), n_items, _ptr(hist2), top2))
        else:
            # the owned solid edges still carry the count stage's in/out flags: $-items the emitter would discard for
            # certain are neither generated nor exchanged (a third of the items; mhb_s2s_extract_edges_pruned)
            cur = self._buf("s_cursor", 8, torch.int64)[:1]
            cur.zero_()
            lib._check(L.mhb_s2s_extract_edges_pruned(_stream(), _ptr(seq_edges), _ptr(aux), n_seqs, n_solid, k, _ptr(sa),
                                                      n_items, _ptr(cur), _ptr(hist2), top2))
            n_items = int(self._to_host(cur)[0])
        own2, n_own2, bounds2, _ = self._partition_and_exchange(sa, n_items, self.W2, top2, hist2, "s", max(n_items, 1),
                                                                 next_byte=self.sbytes[0])
        s_hist = self._first_hist
        if timed:
            self._mark("exchange2")
        srt2 = self._sort_raw(own2, n_own2, self.W2, self.sbytes, "s", s_hist)
        if timed:
            self._mark("s2s_sort")
        wpt = (k + 15) // 16
        cap_b = n_own2 * (4 + 4 * wpt) + 16
        out_bytes = self._buf("sdbg", cap_b, torch.uint8, slack=1.1)
        table = self._buf("table", 65536 * 4, torch.int64)[: 65536 * 4]
        table.zero_()
        totals = self._buf("totals", 16, torch.int64)[:16]
        totals.zero_()
        es = self._buf("s_scratch", L.mhb_s2s_emit_scratch_bytes(n_own2, k), torch.uint8, slack=1.1)
        lib._check(L.mhb_s2s_emit(_stream(), C.c_void_p(srt2), n_own2, k, _ptr(out_bytes), cap_b, _ptr(table), _ptr(totals),
                                  _ptr(es), es.numel()))
        if timed:
            self._mark("s2s")
        return {"n_solid": n_solid, "n_cand": n_cand, "n_mercy": n_mercy, "edges": seq_edges, "mul_hist": mul_hist,
                "bounds": bounds, "bounds2": bounds2, "n_items_sorted": n_own2, "sdbg_bytes": out_bytes, "table": table,
                "totals": totals, "n_records_owned": n_own}


def gather_sdbg_stream(res: dict) -> bytes | None:
    """Canonical SdBG stream of the whole job on rank 0 (validation only)."""
    tot = res["totals"].cpu().numpy()
    nbytes = int(tot[0])
    data = res["sdbg_bytes"][:nbytes].cpu().numpy().tobytes()
    table = res["table"].cpu().numpy().view(np.uint64).reshape(65536, 4)
    mine = lib.sdbg_stream_from_table(table, data)
    objs = [None] * dist.get_world_size()
    dist.all_gather_object(objs, (res["bounds2"].tolist(), mine, int(tot[1])))
    if dist.get_rank() != 0:
        return None
    return b"".join(o[1] for o in objs)  # rank order == bucket order


def _reverse_rows(rows: np.ndarray, read_len: int) -> np.ndarray:
    """`.bin` records (u32 length + packed words) of fixed-length reads -> the same reads reversed (no complement), the
    orientation KmerCounter holds them in and writes to `.cand` (sequence_package.h:284-295, kmer_counter.cpp:387-401)"""
    from . import formats as F
    n = len(rows)
    if n == 0:
        return rows.reshape(0, 1 + (read_len + 15) // 16)
    w = rows[:, 1:].astype(np.uint32)
    idx = np.arange(read_len)
    bases = ((w[:, idx >> 4] >> (30 - 2 * (idx & 15)).astype(np.uint32)) & 3).astype(np.uint8)
    return F.pack_reads_fixed(bases[:, ::-1])


def write_outputs(job: "MultiGpuBuild", res: dict, my_rows: np.ndarray, prefix: str) -> None:
    """The reference's on-disk outputs from a partitioned build (collective): rank r writes `P.edges.<r>` and `P.sdbg.<r>`
    - its contiguous range of the 65 536 buckets, each bucket one contiguous run in exactly one file - and rank 0 the
    merged `P.edges.info` (edge_io_meta.h:25-44: bucket -> file, offset in edges, count), `P.sdbg_info`
    (sdbg_meta.cpp:44-61: records ordered by (file, starting offset), unused ones last), `P.cand` and `P.counting`.
    num_files = world; the consumers are the reference's own readers (edge_reader.h, sdbg_raw_content.cpp:18-95)."""
    world, rank, k, WE = job.world, job.rank, job.k, job.WE
    n_solid = res["n_solid"]
    torch.cuda.synchronize()
    e = res["edges"][: n_solid * WE].cpu().numpy().view(np.uint32).reshape(-1, WE)
    e.tofile(f"{prefix}.edges.{rank}")
    ecnt = np.bincount((e[:, 0] >> 16).astype(np.int64), minlength=65536).astype(np.int64) if n_solid else np.zeros(65536, np.int64)
    tot = res["totals"].cpu().numpy()
    nbytes = int(tot[0])
    res["sdbg_bytes"][:nbytes].cpu().numpy().tofile(f"{prefix}.sdbg.{rank}")
    table = res["table"].cpu().numpy().view(np.uint64).reshape(65536, 4)
    cand_ids = job._bufs["cand"][: res["n_cand"]].cpu().numpy() if res["n_cand"] else np.zeros(0, np.int64)
    cand = _reverse_rows(my_rows[cand_ids], job.read_len).tobytes() if len(cand_ids) else b""
    objs = [None] * world
    dist.all_gather_object(objs, (ecnt, table, cand))
    if rank == 0:
        with open(prefix + ".edges.info", "w") as f:
            n_edges = int(sum(int(o[0].sum()) for o in objs))
            f.write(f"kmer_size {k}\nwords_per_edge {WE}\nnum_files {world}\nnum_buckets 65536\nnum_edges {n_edges}\nis_sorted 1\n")
            off = [np.concatenate([[0], np.cumsum(o[0])[:-1]]) for o in objs]
            owner_of = np.full(65536, -1, np.int64)
            for r, o in enumerate(objs):
                assert (owner_of[o[0] > 0] == -1).all(), "a bucket landed on two ranks"
                owner_of[o[0] > 0] = r
            for b in range(65536):
                r = owner_of[b]
                f.write(f"{b} -1 0 0\n" if r < 0 else f"{b} {r} {int(off[r][b])} {int(objs[r][0][b])}\n")
        with open(prefix + ".sdbg_info", "w") as f:
            wpt = (k + 15) // 16
            f.write(f"k {k}\nwords_per_tip_label {wpt}\nnum_buckets 65536\nnum_files {world}\n")
            used = 0
            for r, o in enumerate(objs):  # rank order, and inside a rank ascending buckets = ascending offsets
                t = o[1]
                for b in np.nonzero(t[:, 1])[0]:
                    f.write(f"{int(b)} {r} {int(t[b, 0])} {int(t[b, 1])} {int(t[b, 2])} {int(t[b, 3])}\n")
                    used += 1
            for _ in range(65536 - used):
                f.write("18446744073709551615 18446744073709551615 0 0 0 0\n")
        with open(prefix + ".cand", "wb") as f:
            for o in objs:  # reads are dealt to the ranks in contiguous blocks: rank order = read order
                f.write(o[2])
        cnt = res["mul_hist"].cpu().numpy()
        with open(prefix + ".counting", "w") as f:
            f.write("".join(f"{i} {int(cnt[i])}\n" for i in range(1, 65536)))
    dist.barrier()


PARITY_CASES = (("syn150_k27", 27), ("syn150_klist", 21), ("syn150_klist", 141), ("polya_k27", 27), ("tandem_k27", 28),
                ("lowcov_k21", 21))


def parity_check(device, cases=PARITY_CASES, verbose=False, files_dir=None) -> dict:
    """Bit-exactness of the partitioned build at the current world size: for every golden case (fixtures minted by the
    unmodified reference, tests/golden) the reads are dealt to the ranks in contiguous blocks, MultiGpuBuild runs its
    normal fused path, and the rank-ordered concatenation of the solid edges, the `.counting` histogram and the
    canonical SdBG stream must reproduce the reference's sha256 digests.  Collective; returns the verdict on every rank."""
    import json
    import os
    from . import formats as F
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    world, rank = dist.get_world_size(), dist.get_rank()
    out = {"world": world, "cases": [], "ok": True}
    for name, k in cases:
        case = os.path.join(root, "tests", "golden", name)
        gold = json.load(open(os.path.join(case, "golden.json")))
        g, m = gold["by_k"][str(k)], gold["m"]
        allw = np.fromfile(os.path.join(case, "reads.lib.bin"), np.uint32)
        rl = int(allw[0])
        stride = 1 + (rl + 15) // 16
        rows = allw.reshape(-1, stride)
        per = (len(rows) + world - 1) // world
        mine = rows[rank * per:(rank + 1) * per]
        bin_dev = torch.from_numpy(np.concatenate([mine.reshape(-1), np.zeros(8, np.uint32)]).view(np.int32)).to(device)
        job = MultiGpuBuild(len(mine), rl, k, m, device, need_mercy=True)
        res = job.run(bin_dev)
        stream = gather_sdbg_stream(res)
        torch.cuda.synchronize()
        edges = res["edges"][: res["n_solid"] * job.WE].cpu().numpy().view(np.uint32).tobytes()
        objs = [None] * world
        dist.all_gather_object(objs, (edges, res["n_solid"], res["n_cand"], res["n_mercy"]))
        verdict = [None]
        if rank == 0:
            cnt = res["mul_hist"].cpu().numpy()
            v = {"case": f"{name}-k{k}",
                 "edges": g["n_solid"] == 0 or F.sha256(b"".join(o[0] for o in objs)) == g["edges_sha256"],
                 "counting": F.sha256("".join(f"{i} {int(cnt[i])}\n" for i in range(1, 65536)).encode()) == g["counting_sha256"],
                 "sdbg": F.sha256(stream) == g["sdbg_sha256"],
                 "n_solid": [int(o[1]) for o in objs], "n_mercy": [int(o[3]) for o in objs]}
            v["ok"] = bool(v["edges"] and v["counting"] and v["sdbg"])
            verdict[0] = v
            if verbose:
                print("parity", v, flush=True)
        if files_dir is not None:
            # file level: every rank writes its own `.edges.<r>` / `.sdbg.<r>`; the canonical streams read back through the
            # bucket tables (formats.py, the reference's reader order) must give the same digests
            prefix = os.path.join(files_dir, f"{name}_k{k}_n{world}")
            write_outputs(job, res, mine, prefix)
            if rank == 0:
                v = verdict[0]
                ce = F.canonical_edges(prefix)
                info, cs, _ = F.canonical_sdbg(prefix)
                v["files"] = bool((g["n_solid"] == 0 or F.sha256(ce.tobytes()) == g["edges_sha256"])
                                  and F.sha256(cs) == g["sdbg_sha256"] and F.file_sha256(prefix + ".cand") == g["cand_sha256"]
                                  and F.file_sha256(prefix + ".counting") == g["counting_sha256"] and info.num_files == world)
                v["prefix"] = prefix
                v["ok"] = bool(v["ok"] and v["files"])
        dist.broadcast_object_list(verdict, src=0)
        out["cases"].append(verdict[0])
        out["ok"] = out["ok"] and verdict[0]["ok"]
        job.close()
        del job, res, bin_dev
    return out


def bench(args, bin_dev, bin_words, rank, world, device, metric, clocks=None):
    """bench.py's N > 1 arm: weak scaling, `args.reads` reads per GPU, one all-to-all per stage."""
    import json
    import os
    import sys

    k, m, n_reads, L = args.k, args.m, args.reads, 150
    # correctness anchor of every N > 1 number: the same fused path on the reference-minted fixtures, before timing
    parity = parity_check(device)
    job = MultiGpuBuild(n_reads, L, k, m, device, need_mercy=True)
    for _ in range(max(1, args.warmup)):
        job.run(bin_dev)
    torch.cuda.synchronize()
    dist.barrier()
    job.times.clear()
    if clocks is not None:
        clocks.start()  # nvidia-smi clocks / throttle reasons of this rank's GPU during the timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = None
    pass_ms = []
    launches0 = lib.launch_count()
    for _ in range(args.steps):
        res = job.run(bin_dev, timed=True)
        # the most recent traced sort over count-width records of this rank's owned count = this step's sort1 (the
        # fused partition pass is not traced; with the NCCL fallback the partitions are, so search instead of counting)
        for back in range(4):
            pm, nrec, words = lib.sort_pass_ms(back)
            if words == job.WR and nrec == res["n_records_owned"] and len(pm) == (2 if job.hashed else len(job.cbytes)):
                pass_ms.append(pm)
                break
        else:
            pass_ms.append(lib.sort_pass_ms(1)[0])  # fused mode: [sort1, sort2] per step
    e1.record()
    launches = (lib.launch_count() - launches0) // max(1, args.steps)
    torch.cuda.synchronize()
    dist.barrier()
    clk = clocks.stop() if clocks is not None else None
    ms = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device=device)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    stage = {}
    names = ["t0", "extract", "c_plan", "exchange1", "sort1", "count", "mercy", "s_plan", "exchange2", "s2s_sort", "s2s"]
    for a, b in zip(names[:-1], names[1:]):
        t = torch.tensor([np.mean([x.elapsed_time(y) for x, y in zip(job.times[a], job.times[b])])], dtype=torch.float64,
                         device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stage[b] = float(t.item())
    own = torch.tensor([res["n_records_owned"], res["n_solid"], res["n_mercy"]], dtype=torch.int64, device=device)
    owns = [torch.zeros_like(own) for _ in range(world)]
    dist.all_gather(owns, own)
    # slowest rank's mean radix pass over the count records
    pm = torch.tensor([float(np.mean([np.mean(x) for x in pass_ms]))], dtype=torch.float64, device=device)
    dist.all_reduce(pm, op=dist.ReduceOp.MAX)

    # ---- e2e: pinned host reads -> device, build, SdBG bytes -> pinned host; device-timed, max over ranks ----
    host_bin = torch.empty(bin_words, dtype=torch.int32).pin_memory()
    host_bin.copy_(bin_dev[:bin_words])
    stage_dev = torch.empty_like(bin_dev)
    out_host = torch.empty(max(1 << 20, int(res["totals"][0].item()) * 2), dtype=torch.uint8).pin_memory()
    e2e_ms = []
    for i in range(1 + max(1, args.e2e_steps)):
        dist.barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        stage_dev[:bin_words].copy_(host_bin, non_blocking=True)
        r2 = job.run(stage_dev)
        nb = int(r2["totals"][0].item())
        out_host[:nb].copy_(r2["sdbg_bytes"][:nb], non_blocking=True)
        tbl = r2["table"].cpu()
        a1.record()
        torch.cuda.synchronize()
        t = torch.tensor([a0.elapsed_time(a1)], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if i > 0:
            e2e_ms.append(float(t.item()))
        del tbl
    nbytes = torch.tensor([nb], dtype=torch.int64, device=device)
    dist.all_reduce(nbytes)
    if rank == 0:
        from .lib import count_record_words
        peak = 6650.0
        src = "fallback (B200_PROFILING.md 6.65 TB/s)"
        pk = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peak, src = float(json.load(open(pk))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        n_edges = world * n_reads * (L - k)
        ms_per_step = float(ms.item())
        S = count_record_words(k) * 4
        n_max = max(int(o[0]) for o in owns)
        ach = 2.0 * n_max * S / (float(pm.item()) * 1e-3) / 1e9
        e2e_v = n_edges / (float(np.mean(e2e_ms)) * 1e-3)
        print(json.dumps({
            "metric": metric, "value": n_edges / (ms_per_step * 1e-3), "unit": "edges/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"synthetic {n_reads}x{L}bp reads PER GPU (30x, 1% subst.), k={k}, m={m}, {world}xB200: "
                                   "top-byte range partition (balanced from the all-reduced histogram), one fused partition+"
                                   "exchange pass per stage storing into the owners' buffers over NVLink (CUDA IPC peer "
                                   "memory), then per-GPU radix sort / count / mercy / seq2sdbg emit",
                       "parallelism": f"bucket-range x{world}", "n_edge_records": n_edges,
                       "records_owned_per_rank": [int(o[0]) for o in owns],
                       "solid_edges_per_rank": [int(o[1]) for o in owns], "mercy_edges_per_rank": [int(o[2]) for o in owns],
                       "l2_note": "inputs (>= 4.9 GB per kernel) exceed the 126 MB L2, no explicit flush needed"},
            "stage_ms_max_over_ranks": stage,
            "roofline": {"bound": "hbm", "kernel": f"k_radix_pass<{S // 4}> (count records, {S} B), slowest rank",
                         "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                         "peak_source": src, "avg_launch_ms": float(pm.item()),
                         "algorithmic_bytes_per_launch": 2 * n_max * S},
            "cpu_baseline": None, "clocks": clk,
            "parity": {"ok": parity["ok"], "world": world, "against": "sha256 digests minted by the unmodified reference "
                       "(tests/golden): edges, .counting, canonical SdBG stream",
                       "cases": [{kk: c[kk] for kk in ("case", "edges", "counting", "sdbg")} for c in parity["cases"]]},
            "e2e": {"value": e2e_v, "unit": "edges/s", "h2d_bytes_per_step": int(world * bin_words * 4),
                    "d2h_bytes_per_step": int(nbytes.item()) + world * 65536 * 32, "ms_per_step": float(np.mean(e2e_ms)),
                    "api": "MultiGpuBuild.run on reads copied from pinned host memory each step; SdBG bytes + bucket "
                           "table copied back to pinned host memory"},
            "gpu_launches": int(launches),
        }))
    sys.stdout.flush()
    torch.cuda.synchronize()
    job.close()
    dist.barrier()
    dist.destroy_process_group()
    if not parity["ok"]:
        raise SystemExit("multi-GPU parity check FAILED: " + json.dumps(parity["cases"]))
