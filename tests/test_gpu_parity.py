"""GPU parity tests: the CUDA path (through the C ABI) against the oracle on the same inputs, against
the golden fixtures minted by the unmodified reference, and - at sizes the oracle cannot reach in
seconds - through size-independent properties.  Integer/byte work: every comparison is bit-exact."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
from megahit_b200 import formats as F
from megahit_b200 import lib, synth

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _oracle():
    import oracle_pipeline as OP
    from oracle import oracle as O
    return OP, O


# ------------------------------------------------------------------------------------------------
# A4: the radix sort on its own
# ------------------------------------------------------------------------------------------------
def _np_lsd(recs, sort_bytes):
    w = recs.shape[1]
    order = np.arange(len(recs))
    for b in sort_bytes:
        digit = (recs[order, w - 1 - (b >> 2)] >> (8 * (b & 3))) & 255
        order = order[np.argsort(digit, kind="stable")]
    return recs[order]


@pytest.mark.parametrize("words,n,nbytes", [(1, 1000, 4), (2, 1, 8), (2, 6911, 7), (2, 6913, 7), (2, 300_000, 7),
                                            (3, 250_000, 10), (4, 100_001, 16), (5, 70_000, 3), (9, 20_000, 36),
                                            (17, 5_000, 20), (2, 2_000_000, 8)])
def test_sort_records_matches_stable_lsd(words, n, nbytes):
    torch = _torch()
    from megahit_b200 import dev
    rng = np.random.default_rng(words * 1000 + n)
    recs = rng.integers(0, 2 ** 32, size=(n, words), dtype=np.uint64).astype(np.uint32)
    # few distinct values in the sorted bytes -> long ties, so stability is actually exercised
    if n > 10:
        recs[:, 0] &= np.uint32(0x0F0F0F0F)
    all_bytes = list(range(4 * words))
    sort_bytes = sorted(rng.choice(all_bytes, size=min(nbytes, len(all_bytes)), replace=False).tolist())
    a = torch.from_numpy(recs.view(np.int32).reshape(-1).copy()).cuda()
    a = torch.cat([a, torch.zeros(4, dtype=torch.int32, device="cuda")])
    b = torch.empty_like(a)
    out = dev.sort_records(a, b, n, words, sort_bytes)
    got = out[: n * words].cpu().numpy().view(np.uint32).reshape(n, words)
    exp = _np_lsd(recs, sort_bytes)
    assert (got == exp).all()


def test_sort_skewed_digits():
    """all records share every digit but one (poly-A like skew) + a run of equal keys longer than a tile"""
    torch = _torch()
    from megahit_b200 import dev
    n = 200_000
    recs = np.zeros((n, 2), np.uint32)
    recs[:, 1] = np.arange(n, dtype=np.uint32)[::-1] % 7  # payload-ish low bits, not sorted
    recs[50_000:60_000, 0] = 0xFFFFFFFF
    recs[::3, 0] = 1 << 8
    sort_bytes = [1, 2, 3, 4, 5, 6, 7]
    a = torch.from_numpy(np.concatenate([recs.view(np.int32).reshape(-1), np.zeros(4, np.int32)])).cuda()
    out = dev.sort_records(a, torch.empty_like(a), n, 2, sort_bytes)
    got = out[: n * 2].cpu().numpy().view(np.uint32).reshape(n, 2)
    assert (got == _np_lsd(recs, sort_bytes)).all()


@pytest.mark.parametrize("words,n,sort_bytes", [(2, 1, [1, 2, 3]), (2, 4607, [1, 2, 3, 4, 5, 6, 7]),
                                                  (2, 6912 * 3 + 1, [1, 2, 3, 4, 5, 6, 7]), (2, 400_003, [1, 2, 3, 4, 5, 6, 7]),
                                                  (3, 3071, [2, 5, 11]), (3, 200_001, [0, 1, 2, 4, 5, 6, 7, 8, 9, 10]),
                                                  (4, 3840 * 2 + 1, [0, 6, 13]), (5, 30_011, [3, 9, 17]),
                                                  (17, 768 * 5 + 7, [1, 40, 67])])
def test_sort_ragged_and_single_tiles(words, n, sort_bytes):
    """the stable LSD order with ragged last tiles and single-tile inputs (tiles of 6912, 4608, 3840, 2304 and 768
    records at 2, 3, 4, 5 and 17 words)"""
    torch = _torch()
    from megahit_b200 import dev
    rng = np.random.default_rng(words * 1_000_003 + n)
    recs = rng.integers(0, 2 ** 32, size=(n, words), dtype=np.uint64).astype(np.uint32)
    recs[:, 0] &= np.uint32(0x0F0F0F0F)
    a = torch.from_numpy(np.concatenate([recs.view(np.int32).reshape(-1), np.zeros(4, np.int32)])).cuda()
    out = dev.sort_records(a, torch.empty_like(a), n, words, sort_bytes)
    got = out[: n * words].cpu().numpy().view(np.uint32).reshape(n, words)
    assert (got == _np_lsd(recs, sort_bytes)).all()


# ------------------------------------------------------------------------------------------------
# count + seq2sdbg on every golden case: CUDA == oracle == reference digests
# ------------------------------------------------------------------------------------------------
def _gpu_count(case, k, m):
    bin_words = np.fromfile(os.path.join(case, "reads.lib.bin"), np.uint32)
    _, n_reads = F.read_lib_info(os.path.join(case, "reads.lib"))
    return lib.count_host(bin_words, n_reads, k, m, want_mercy=True)


@pytest.mark.parametrize("name,k,m,gold", golden_cases())
def test_count_and_sdbg_match_oracle_and_reference(name, k, m, gold):
    OP, O = _oracle()
    case = os.path.join(GOLDEN, name)
    reads = OP.load_reads(case)
    oc = OP.oracle_count(reads, k, m)
    g = _gpu_count(case, k, m)
    assert g["n_edge_records"] == oc["n_records"]
    assert g["n_solid"] == oc["n_solid"] == gold["n_solid"]
    assert (g["edges"] == oc["edges"]).all()
    assert F.sha256(g["edges"].tobytes()) == gold["edges_sha256"]
    assert (g["counting"] == oc["counting"]).all()
    assert F.sha256(O.counting_text(g["counting"])) == gold["counting_sha256"]
    assert (g["cand_ids"] == oc["cand_ids"]).all()
    assert F.sha256(reads.bin_bytes(g["cand_ids"])) == gold["cand_sha256"]

    # seq2sdbg on the same sequences the reference would load: edges + mercy edges (host logic under test
    # separately in test_file_level_*), so this isolates S-extract / sort / S-emit
    seqs, mult = O.edges_as_seqs(oc["edges"], k)
    cand = O.unpack_bin(oc["cand_bytes"], reverse=False)
    me = O.gen_mercy(oc["edges"], cand, k)
    if len(me):
        seqs = O.Seqs.concat([seqs, O.Seqs.from_fixed(me, k + 1)])
        mult = np.concatenate([mult, np.ones(len(me), np.uint16)])
    os_ = O.seq2sdbg(seqs, mult, k)
    gs = lib.s2s_host(seqs.words, seqs.word_off, seqs.len, mult, k)
    assert gs["n_records"] == os_["n_records"]
    assert gs["n_items"] == os_["n_items"] == gold["sdbg_items"]
    assert gs["n_tips"] == int(os_["bucket_tips"].sum()) == gold["sdbg_tips"]
    assert gs["n_large_mul"] == int(os_["bucket_large_mul"].sum()) == gold["sdbg_large_mul"]
    assert gs["bytes"] == os_["bytes"]
    assert (gs["bucket_table"][:, 1] == os_["bucket_items"]).all()
    assert (gs["bucket_table"][:, 2] == os_["bucket_tips"]).all()
    assert (gs["bucket_table"][:, 3] == os_["bucket_large_mul"]).all()
    nz = os_["bucket_items"] > 0
    assert (gs["bucket_table"][nz, 0] == os_["bucket_byte_off"][:-1][nz]).all()
    assert (gs["w_count"] == os_["w_count"]).all() and gs["ones_in_last"] == os_["ones_in_last"]
    assert F.sha256(lib.sdbg_stream_from_table(gs["bucket_table"], gs["bytes"])) == gold["sdbg_sha256"]


# ------------------------------------------------------------------------------------------------
# fused build (count -> device mercy edges -> seq2sdbg, nothing leaves HBM in between)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k,m,gold", [c for c in golden_cases() if c.values[0] in ("toy_k21", "syn150_k27", "synvar_k21_m3", "synvar_k31_m1", "polya_k27")])
@pytest.mark.parametrize("div", [3, 17])
def test_count_in_rounds_matches_one_pass(name, k, m, gold, div):
    """A13: the count stage run in rounds over leading-byte ranges (forced by capping the round size) gives the
    edges / `.cand` ids / `.counting` of the single pass and of the reference"""
    case = os.path.join(GOLDEN, name)
    one = _gpu_count(case, k, m)
    n = int(one["n_edge_records"])
    if n == 0:
        pytest.skip("no edges")
    bin_words = np.fromfile(os.path.join(case, "reads.lib.bin"), np.uint32)
    _, n_reads = F.read_lib_info(os.path.join(case, "reads.lib"))
    limit = max(1, n // div)
    lib.set_round_limit(limit)
    try:
        try:
            g = lib.count_host(bin_words, n_reads, k, m, want_mercy=True)
        except lib.MhbError as e:
            # a single leading byte may hold more than the cap (poly-A): that must be reported, not mis-sorted
            assert "more than one round can take" in str(e)
            return
    finally:
        lib.set_round_limit(0)
    assert g["n_rounds"] > 1
    assert g["n_solid"] == one["n_solid"] and (g["edges"] == one["edges"]).all()
    assert (g["counting"] == one["counting"]).all()
    assert (g["cand_ids"] == one["cand_ids"]).all() and g["n_has_tips"] == one["n_has_tips"]
    assert F.sha256(g["edges"].tobytes()) == gold["edges_sha256"]


@pytest.mark.parametrize("name,k,m,gold", golden_cases())
def test_fused_build_matches_reference(name, k, m, gold):
    OP, O = _oracle()
    case = os.path.join(GOLDEN, name)
    bin_words = np.fromfile(os.path.join(case, "reads.lib.bin"), np.uint32)
    _, n_reads = F.read_lib_info(os.path.join(case, "reads.lib"))
    g = lib.build_host(bin_words, n_reads, k, m, need_mercy=True, want_edges=True)
    assert g["n_solid"] == gold["n_solid"]
    if gold["n_solid"]:
        assert F.sha256(g["edges"].tobytes()) == gold["edges_sha256"]
    reads = OP.load_reads(case)
    assert F.sha256(reads.bin_bytes(g["cand_ids"])) == gold["cand_sha256"]
    assert F.sha256(O.counting_text(g["counting"])) == gold["counting_sha256"]
    # mercy edges: same multiset as the oracle's GenMercyEdges (order is irrelevant downstream)
    oc = OP.oracle_count(reads, k, m)
    cand = O.unpack_bin(oc["cand_bytes"], reverse=False)
    assert g["n_mercy"] == len(O.gen_mercy(oc["edges"], cand, k))
    assert g["n_items"] == gold["sdbg_items"] and g["n_tips"] == gold["sdbg_tips"]
    assert g["n_large_mul"] == gold["sdbg_large_mul"]
    assert F.sha256(lib.sdbg_stream_from_table(g["bucket_table"], g["bytes"])) == gold["sdbg_sha256"]


@pytest.mark.parametrize("name,k", [("syn150_k27", 27), ("toy_k21", 21), ("lowcov_k21", 21), ("synvar_k21_m3", 21), ("syn150_klist", 59)])
def test_fused_build_in_rounds_matches_reference(name, k):
    """A13 for the fused build: with round caps set (or when the resident plan does not fit) mhb_build_host runs count ->
    mercy edges -> seq2sdbg stage by stage, each in rounds over bucket ranges; same edges / `.cand` / SdBG bytes"""
    gold_case = [c for c in golden_cases() if c.id == f"{name}-k{k}"][0]
    m, gold = gold_case.values[2], gold_case.values[3]
    case = os.path.join(GOLDEN, name)
    bin_words = np.fromfile(os.path.join(case, "reads.lib.bin"), np.uint32)
    _, n_reads = F.read_lib_info(os.path.join(case, "reads.lib"))
    one = lib.build_host(bin_words, n_reads, k, m, need_mercy=True)
    lib.set_round_limit(max(1, int(one["n_edge_records"]) // 4))
    lib.set_s2s_round_limit(max(1, int(one["n_solid"] + one["n_mercy"]) * 6 // 4))
    try:
        try:
            g = lib.build_host(bin_words, n_reads, k, m, need_mercy=True, want_edges=True)
        except lib.MhbError as e:  # a single bucket above the cap is reported, never mis-sorted
            assert "round" in str(e)
            return
    finally:
        lib.set_round_limit(0)
        lib.set_s2s_round_limit(0)
    assert g["n_solid"] == gold["n_solid"] and g["n_mercy"] == one["n_mercy"]
    if gold["n_solid"]:
        assert F.sha256(g["edges"].tobytes()) == gold["edges_sha256"]
    assert g["n_items"] == gold["sdbg_items"] and g["n_tips"] == gold["sdbg_tips"]
    assert F.sha256(lib.sdbg_stream_from_table(g["bucket_table"], g["bytes"])) == gold["sdbg_sha256"]


def test_fused_build_into_caller_buffer():
    case = os.path.join(GOLDEN, "syn150_k27")
    gold = [c for c in golden_cases() if c.id == "syn150_k27-k27"][0].values[3]
    bin_words = np.fromfile(os.path.join(case, "reads.lib.bin"), np.uint32)
    buf = np.zeros(4 << 20, np.uint8)
    g = lib.build_host(bin_words, 3000, 27, 2, need_mercy=True, sdbg_out=buf, copy_bytes=False)
    assert F.sha256(lib.sdbg_stream_from_table(g["bucket_table"], buf[: g["n_bytes"]].tobytes())) == gold["sdbg_sha256"]


# ------------------------------------------------------------------------------------------------
# file level: the sub-commands on the reference's on-disk formats (incl. host-side mercy + writers)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k,m,gold", [c for c in golden_cases()
                                            if c.id in ("toy_k21-k21", "syn150_k27-k27", "synvar_k31_m1-k31",
                                                        "empty_k21-k21", "polya_k27-k27", "syn150_klist-k141")])
def test_file_level_subcommands_match_reference(name, k, m, gold, tmp_path):
    case = os.path.join(GOLDEN, name)
    p = str(tmp_path / f"k{k}")
    lib.count_run(os.path.join(case, "reads.lib"), p, k=k, m=m, host_mem=1e9, num_cpu_threads=2)
    lib.seq2sdbg_run(p, k=k, input_prefix=p, need_mercy=True, host_mem=1e9, num_cpu_threads=2)
    edges = F.canonical_edges(p)
    assert len(edges) == gold["n_solid"]
    if gold["n_solid"]:
        assert F.sha256(edges.tobytes()) == gold["edges_sha256"]
    assert F.file_sha256(p + ".cand") == gold["cand_sha256"]
    assert F.file_sha256(p + ".counting") == gold["counting_sha256"]
    info, stream, table = F.canonical_sdbg(p)
    assert info.k == gold["sdbg_k"] and info.words_per_tip_label == gold["sdbg_words_per_tip_label"]
    assert int(table[:, 0].sum()) == gold["sdbg_items"] and int(table[:, 1].sum()) == gold["sdbg_tips"]
    assert F.sha256(stream) == gold["sdbg_sha256"]


def test_cli_binary_runs_count(tmp_path):
    """the drop-in `megahit_core` executable: same argv as src/megahit:783-803 builds"""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "megahit_b200", "bin", "megahit_core")
    case = os.path.join(GOLDEN, "toy_k21")
    gold = [c for c in golden_cases() if c.id == "toy_k21-k21"][0].values[3]
    p = str(tmp_path / "21")
    r = subprocess.run([exe, "count", "-k", "21", "-m", "2", "--host_mem", "1e9", "--mem_flag", "1", "--output_prefix", p,
                        "--num_cpu_threads", "2", "--read_lib_file", os.path.join(case, "reads.lib")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Total number of solid edges: %d" % gold["n_solid"] in r.stderr
    r = subprocess.run([exe, "seq2sdbg", "--host_mem", "1e9", "--mem_flag", "1", "--output_prefix", p,
                        "--num_cpu_threads", "2", "-k", "21", "--kmer_from", "0", "--input_prefix", p, "--need_mercy"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert F.sha256(F.canonical_sdbg(p)[1]) == gold["sdbg_sha256"]
    assert subprocess.run([exe, "checkcpu"], capture_output=True, text=True).stdout.strip() == "1"
    assert subprocess.run([exe, "kmax"], capture_output=True, text=True).stdout.strip() == "255"
    bad = subprocess.run([exe, "count", "-k", "21"], capture_output=True, text=True)
    assert bad.returncode == 1 and "No read library configuration file!" in bad.stderr


# ------------------------------------------------------------------------------------------------
# medium size: oracle still finishes in seconds
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [27, 59])
def test_medium_synthetic_against_oracle(k):
    OP, O = _oracle()
    n_reads = 40_000
    b = synth.synth_reads(n_reads, 150, 200_000, 0.01, seed=123)
    reads = O.unpack_bin(b.tobytes(), reverse=True)
    oc = OP.oracle_count(reads, k, 2)
    g = lib.count_host(b.reshape(-1), n_reads, k, 2)
    assert g["n_solid"] == oc["n_solid"] and (g["edges"] == oc["edges"]).all()
    assert (g["counting"] == oc["counting"]).all() and (g["cand_ids"] == oc["cand_ids"]).all()
    seqs, mult = O.edges_as_seqs(oc["edges"], k)
    os_ = O.seq2sdbg(seqs, mult, k)
    gs = lib.s2s_host(seqs.words, seqs.word_off, seqs.len, mult, k)
    assert gs["bytes"] == os_["bytes"] and gs["n_items"] == os_["n_items"]


# ------------------------------------------------------------------------------------------------
# large size: properties that do not need the oracle
# ------------------------------------------------------------------------------------------------
def test_large_synthetic_properties():
    """2 M x 150 bp, k=27 (246 M edge records): sortedness, conservation of occurrences, idempotence."""
    torch = _torch()
    from megahit_b200 import dev
    n_reads, L, k, m = 2_000_000, 150, 27, 2
    bin_dev = synth.synth_reads_torch(n_reads, L, 10_000_000, 0.01, 99, "cuda").reshape(-1)
    bin_dev = torch.cat([bin_dev, torch.zeros(8, dtype=torch.int32, device="cuda")])
    plan = dev.CountPlan(n_reads, L, k, m, "cuda", want_mercy=True, mode="sort")
    n_solid = plan.run(bin_dev)
    edges = plan.edges_host(n_solid)
    hist = plan.mul_hist.cpu().numpy()
    n_rec = n_reads * (L - k)
    # every occurrence is counted exactly once (no multiplicity saturates at this coverage)
    assert hist[65535] == 0 and int((hist * np.arange(65536)).sum()) == n_rec
    assert n_solid == int(hist[m:].sum())
    # strictly ascending canonical (k+1)-mers; multiplicities consistent with the histogram
    key = (edges[:, 0].astype(np.uint64) << np.uint64(32)) | edges[:, 1].astype(np.uint64)
    assert (key[1:] > key[:-1]).all()
    assert (edges[:, 1] & 0xFF == 0).all()
    mult = edges[:, 2] & 0xFFFF
    assert (np.bincount(mult, minlength=65536)[m:] == hist[m:]).all()
    # the sorted records themselves: non-decreasing on the key bytes, and a permutation of the extraction
    hi = plan.sorted[: plan.n * 2].view(-1, 2)
    k64 = ((hi[:, 0].to(torch.int64) & 0xFFFFFFFF) << 24) | ((hi[:, 1].to(torch.int64) & 0xFFFFFFFF) >> 8)
    assert bool((k64[1:] >= k64[:-1]).all())
    # idempotence: a second run over the same resident library gives the same bytes
    first = edges.copy()
    n2 = plan.run(bin_dev)
    assert n2 == n_solid and (plan.edges_host(n2) == first).all()
    # mercy arrays: candidates exist and respect last > first
    f = plan.first[:n_reads].cpu().numpy().view(np.uint32)
    l = plan.last[:n_reads].cpu().numpy().view(np.uint32)
    both = (f != 0xFFFFFFFF) & (l != 0xFFFFFFFF)
    assert both.sum() > 0 and (f[f != 0xFFFFFFFF] <= L - k).all() and (l[l != 0xFFFFFFFF] <= L - k - 1).all()
    # the partition + hash-aggregation count stage on the same library: identical edges, flags, histogram, mercy marks
    aux = plan.aux[:n_solid].cpu().numpy().copy()
    del plan
    torch.cuda.empty_cache()
    hp = dev.CountPlan(n_reads, L, k, m, "cuda", want_mercy=True, mode="hashed")
    assert hp.run(bin_dev) == n_solid
    assert (hp.edges_host(n_solid) == first).all() and (hp.aux[:n_solid].cpu().numpy() == aux).all()
    assert (hp.mul_hist.cpu().numpy() == hist).all()
    assert (hp.first[:n_reads].cpu().numpy().view(np.uint32) == f).all() and (hp.last[:n_reads].cpu().numpy().view(np.uint32) == l).all()


# ------------------------------------------------------------------------------------------------
# A11 through the host-level ABI, and the multi-GPU building blocks on one GPU
# ------------------------------------------------------------------------------------------------
def _bare_kmers(a, k, bare=False):
    """sorted (k+1)-mers of mercy edges: `.edges`-format records (multiplicity 1 in the low 16 bits of the last word,
    seq_to_sdbg.cpp:354) or, bare=True, the oracle's plain packed (k+1)-mers"""
    a = np.ascontiguousarray(a, np.uint32).reshape(len(a), -1).copy()
    wm = (k + 1 + 15) // 16
    if not bare:
        assert ((a[:, -1] & 0xFFFF) == 1).all()
        a[:, -1] &= np.uint32(0xFFFF0000)
        assert (a[:, wm:] == 0).all()
    return sorted(map(bytes, np.ascontiguousarray(a[:, :wm])))


@pytest.mark.parametrize("name,k,m,gold", [c for c in golden_cases() if c.values[0] in ("toy_k21", "syn150_k27", "synvar_k31_m1", "lowcov_k21")])
def test_mercy_host_matches_oracle(name, k, m, gold):
    """mhb_mercy_host (what `seq2sdbg --need_mercy` calls): sorted `.edges` records + the `.cand` image -> the same
    multiset of mercy edges as the oracle's GenMercyEdges"""
    OP, O = _oracle()
    reads = OP.load_reads(os.path.join(GOLDEN, name))
    oc = OP.oracle_count(reads, k, m)
    cand = O.unpack_bin(oc["cand_bytes"], reverse=False)
    exp = O.gen_mercy(oc["edges"], cand, k)
    got = lib.mercy_host(k, oc["edges"], np.frombuffer(oc["cand_bytes"], np.uint32))
    assert len(got) == len(exp)
    if len(exp):
        assert _bare_kmers(got, k) == _bare_kmers(exp, k, bare=True)


def test_plan_partition_kernel_matches_host_planner():
    """mhb_plan_partition (device) == multigpu.plan_ranges / split_counts (host model, also exercised over gloo)"""
    torch = _torch()
    import ctypes as C
    from megahit_b200 import multigpu
    L = lib.load()
    rng = np.random.default_rng(3)
    for world in (1, 2, 3, 4, 8, 16):
        for rank in {0, world // 2, world - 1}:
            hist = rng.integers(0, 5000, (world, 256)).astype(np.int64)
            hist[:, : rng.integers(0, 100)] //= 50  # skew
            bounds = multigpu.plan_ranges(hist.sum(0), world)
            send = np.stack([multigpu.split_counts(hist[r], bounds) for r in range(world)])  # [src][owner]
            h = torch.from_numpy(hist.reshape(-1)).cuda()
            lut = torch.zeros(256, dtype=torch.uint8, device="cuda")
            addr = torch.zeros(256, dtype=torch.int64, device="cuda")
            plan = torch.zeros(64, dtype=torch.int64, device="cuda")
            base = [(o + 1) << 40 for o in range(world)]
            peers = (C.c_uint64 * 16)(*base)
            lib._check(L.mhb_plan_partition(None, C.c_void_p(h.data_ptr()), world, rank, 12, peers, C.c_void_p(lut.data_ptr()),
                                            C.c_void_p(addr.data_ptr()), C.c_void_p(plan.data_ptr())))
            p = plan.cpu().numpy()
            assert (p[32:33 + world] == bounds).all(), (world, p[32:33 + world], bounds)
            assert (p[:world] == send.sum(0)).all() and (p[16:16 + world] == send[rank]).all()
            owner = np.repeat(np.arange(world), np.diff(bounds))
            assert (lut.cpu().numpy() == owner).all()
            exp_addr = [base[o] + int(send[:rank, o].sum()) * 12 for o in range(world)]
            assert addr.cpu().numpy()[:world].tolist() == exp_addr


@pytest.mark.parametrize("name,k,m,gold", [c for c in golden_cases() if c.values[0] in ("syn150_k27", "lowcov_k21", "toy_k21")])
@pytest.mark.parametrize("n_owner", [1, 3])
def test_owner_answered_mercy_search_matches_single_segment(name, k, m, gold, n_owner):
    """the multi-GPU form of the mercy search on one GPU: the edge array cut into n_owner leading-byte ranges, every
    "rank" answering only the searches that land in its range (mhb_mercy_probe_owned), the answer planes OR-ed
    (mhb_mercy_count_planes) -> the same mercy edges as the ordinary single-segment search"""
    torch = _torch()
    import ctypes as C
    OP, O = _oracle()
    L = lib.load()
    case = os.path.join(GOLDEN, name)
    reads = OP.load_reads(case)
    oc = OP.oracle_count(reads, k, m)
    cand_reads = O.unpack_bin(oc["cand_bytes"], reverse=False)
    exp = np.asarray(O.gen_mercy(oc["edges"], cand_reads, k), np.uint32)
    n_cand = len(oc["cand_ids"])
    if n_cand == 0:
        pytest.skip("no candidates")
    binw = np.fromfile(os.path.join(case, "reads.lib.bin"), np.uint32)
    _, n_reads = F.read_lib_info(os.path.join(case, "reads.lib"))
    # variable-length layout arrays (works for fixed-length libraries too)
    rec_off, edge_off, pos, e, mx = [], [], 0, 0, 0
    for _ in range(n_reads):
        Lr = int(binw[pos])
        rec_off.append(pos)
        edge_off.append(e)
        e += max(0, Lr - k)
        mx = max(mx, Lr)
        pos += 1 + (Lr + 15) // 16
    rec_off.append(pos)
    edge_off.append(e)
    d_bin = torch.from_numpy(np.concatenate([binw, np.zeros(8, np.uint32)]).view(np.int32)).cuda()
    d_ro = torch.tensor(rec_off, dtype=torch.int64, device="cuda")
    d_eo = torch.tensor(edge_off, dtype=torch.int64, device="cuda")
    d_ids = torch.from_numpy(oc["cand_ids"].astype(np.int64)).cuda()
    rd = lib.DevReads(d_bin.data_ptr(), len(binw), n_reads, 0, d_ro.data_ptr(), d_eo.data_ptr())
    we = lib.words_per_edge(k)
    edges = np.ascontiguousarray(oc["edges"], np.uint32).reshape(-1, we)
    top = edges[:, 0] >> 24
    cuts = [0] + [int(np.quantile(top, q)) + 1 for q in np.linspace(0, 1, n_owner + 1)[1:-1]] + [256]
    cuts = sorted(set(cuts))
    n_own = len(cuts) - 1
    owner = np.zeros(256, np.uint8)
    for o in range(n_own):
        owner[cuts[o]:cuts[o + 1]] = o
    owner_c = (C.c_uint8 * 256)(*owner.tolist())
    pw = L.mhb_mercy_planes_words(n_cand, mx)
    planes = torch.zeros(n_own * pw, dtype=torch.int32, device="cuda")
    keep = []
    for o in range(n_own):
        seg = edges[owner[top] == o]
        d_seg = torch.from_numpy(np.concatenate([seg.reshape(-1), np.zeros(4, np.uint32)]).view(np.int32)).cuda()
        lut = torch.empty(L.mhb_edge_lut_bytes(), dtype=torch.uint8, device="cuda")
        lib._check(L.mhb_edge_lut_build(None, C.c_void_p(d_seg.data_ptr()), len(seg), k, C.c_void_p(lut.data_ptr())))
        lib._check(L.mhb_mercy_probe_owned(None, C.byref(rd), C.c_void_p(d_ids.data_ptr()), n_cand, mx, k,
                                           C.c_void_p(d_seg.data_ptr()), len(seg), C.c_void_p(lut.data_ptr()), owner_c, o,
                                           C.c_void_p(planes.data_ptr() + o * pw * 4)))
        keep.append((d_seg, lut))
    scratch = torch.empty(L.mhb_mercy_edges_scratch_bytes(n_cand, mx), dtype=torch.uint8, device="cuda")
    nm = C.c_uint64(0)
    lib._check(L.mhb_mercy_count_planes(None, C.byref(rd), C.c_void_p(d_ids.data_ptr()), n_cand, mx, k,
                                        C.c_void_p(planes.data_ptr()), n_own, pw, C.byref(nm), C.c_void_p(scratch.data_ptr()),
                                        scratch.numel()))
    assert nm.value == len(exp)
    out = torch.zeros(max(1, nm.value) * we, dtype=torch.int32, device="cuda")
    lib._check(L.mhb_mercy_edges_write(None, C.byref(rd), C.c_void_p(d_ids.data_ptr()), n_cand, mx, k, C.c_void_p(out.data_ptr()),
                                       nm.value, nm.value, C.c_void_p(scratch.data_ptr()), scratch.numel()))
    got = out.cpu().numpy().view(np.uint32)[: nm.value * we].reshape(-1, we)
    assert _bare_kmers(got, k) == _bare_kmers(exp.reshape(len(exp), -1), k, bare=True)


# ------------------------------------------------------------------------------------------------
# A4 + A5 by partition + per-bucket hash aggregation == sort + run-length count
# ------------------------------------------------------------------------------------------------
def _count_both_ways(recs: np.ndarray, k: int, m: int):
    """recs: (n, 2) uint32 count records.  Returns ((edges, aux, hist, n_solid) sorted path, same for the hashed path)."""
    torch = _torch()
    import ctypes as C
    from megahit_b200 import dev
    L = lib.load()
    n = len(recs)
    we = lib.words_per_edge(k)
    cap = n // max(1, m) + 1
    out = []
    for hashed in (False, True):
        a = torch.from_numpy(np.concatenate([recs.reshape(-1), np.zeros(4, np.uint32)]).view(np.int32)).cuda()
        b = torch.empty_like(a)
        edges = torch.zeros(cap * we + 4, dtype=torch.int32, device="cuda")
        aux = torch.zeros(cap + 4, dtype=torch.uint8, device="cuda")
        hist = torch.zeros(65536, dtype=torch.int64, device="cuda")
        ns = torch.zeros(8, dtype=torch.int64, device="cuda")
        if hashed:
            ws = torch.empty(L.mhb_count_hashed_workspace_bytes(n, k, m), dtype=torch.uint8, device="cuda")
            lib._check(L.mhb_count_solid_hashed(None, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), n, k, m, None,
                                                C.c_void_p(edges.data_ptr()), C.c_void_p(aux.data_ptr()), cap,
                                                C.c_void_p(hist.data_ptr()), C.c_void_p(ns.data_ptr()), C.c_void_p(ws.data_ptr()),
                                                ws.numel()))
        else:
            srt = dev.sort_records(a, b, n, 2, lib.count_sort_bytes(k))
            sc = torch.empty(L.mhb_count_solid_scratch_bytes(n), dtype=torch.uint8, device="cuda")
            lib._check(L.mhb_count_solid(None, C.c_void_p(srt.data_ptr()), n, k, m, C.c_void_p(edges.data_ptr()),
                                         C.c_void_p(aux.data_ptr()), cap, C.c_void_p(hist.data_ptr()), C.c_void_p(ns.data_ptr()),
                                         C.c_void_p(sc.data_ptr()), sc.numel()))
        torch.cuda.synchronize()
        n_solid = int(ns[0].item())
        out.append((edges[: n_solid * we].cpu().numpy().copy(), aux[:n_solid].cpu().numpy().copy(), hist.cpu().numpy().copy(), n_solid))
    return out


@pytest.mark.parametrize("case", ["reads30x", "all_distinct", "one_bucket_many_keys", "one_key_huge", "few_keys_high_mult",
                                  "k21_reads", "m1", "m5", "tiny"])
def test_hashed_count_matches_sort_and_count(case):
    """mhb_count_solid_hashed (2 partition passes + per-bucket hash aggregation) gives the edges, aux flags, multiplicity
    histogram and solid count of the full sort + mhb_count_solid, on real extractions and on adversarial key sets: a bucket
    with more distinct keys than the table holds (sub-range retries), one key repeated beyond the 16-bit tally fields
    (clamping between chunks), multiplicities above the shared-memory histogram"""
    torch = _torch()
    import ctypes as C
    import zlib
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    k, m = 27, 2

    def from_reads(n_reads, kk, genome):
        b = synth.synth_reads_torch(n_reads, 150, genome, 0.01, 5, "cuda").reshape(-1)
        b = torch.cat([b, torch.zeros(8, dtype=torch.int32, device="cuda")])
        n = n_reads * (150 - kk)
        a = torch.empty(n * 2 + 4, dtype=torch.int32, device="cuda")
        rd = lib.DevReads(b.data_ptr(), b.numel(), n_reads, 150, None, None)
        lib._check(lib.load().mhb_count_extract(None, C.byref(rd), kk, C.c_void_p(a.data_ptr()), n, None, 0))
        return a[: n * 2].cpu().numpy().view(np.uint32).reshape(n, 2)

    def with_pn(keys):  # keys: uint64 with the low 8 bits free -> records with random prev/next (0..4 each)
        pn = (rng.integers(0, 5, len(keys)) << 3 | rng.integers(0, 5, len(keys))).astype(np.uint64)
        v = (keys & ~np.uint64(0xFF)) | pn
        return np.stack([(v >> np.uint64(32)).astype(np.uint32), (v & np.uint64(0xFFFFFFFF)).astype(np.uint32)], axis=1)

    if case == "reads30x":
        recs = from_reads(150_000, 27, 750_000)
    elif case == "k21_reads":
        k = 21
        recs = from_reads(60_000, 21, 300_000)
    elif case == "m1":
        m = 1
        recs = from_reads(20_000, 27, 100_000)
    elif case == "m5":
        m = 5
        recs = from_reads(60_000, 27, 200_000)
    elif case == "all_distinct":
        recs = with_pn(rng.integers(0, 2 ** 63, 400_000, dtype=np.uint64) << np.uint64(1))
    elif case == "one_bucket_many_keys":  # 60 k distinct keys in ONE 16-bit bucket, each 1..3 times
        base = rng.integers(0, 2 ** 40, 60_000, dtype=np.uint64) << np.uint64(8) | (np.uint64(0x1234) << np.uint64(48))
        recs = with_pn(np.repeat(base, rng.integers(1, 4, len(base))))
    elif case == "one_key_huge":  # one key 200 k times (> 65535: tally clamp) + noise in the same bucket
        hot = np.full(200_000, (0x00FF << 48) | (0xABCDEF << 8), np.uint64)
        noise = rng.integers(0, 2 ** 40, 5_000, dtype=np.uint64) << np.uint64(8) | (np.uint64(0x00FF) << np.uint64(48))
        recs = with_pn(np.concatenate([hot, noise]))
    elif case == "few_keys_high_mult":  # multiplicities 1000..3000: above the shared-memory histogram range
        base = rng.integers(0, 2 ** 55, 300, dtype=np.uint64) << np.uint64(8)
        recs = with_pn(np.repeat(base, rng.integers(1000, 3000, len(base))))
    else:  # tiny
        recs = with_pn(np.array([5 << 8, 5 << 8, 7 << 8], np.uint64))
    recs = recs[rng.permutation(len(recs))]
    (e0, a0, h0, n0), (e1, a1, h1, n1) = _count_both_ways(recs, k, m)
    assert n0 == n1 and (n0 > 0 or case == "all_distinct")
    assert (e0 == e1).all() and (a0 == a1).all() and (h0 == h1).all()


@pytest.mark.parametrize("words,n", [(2, 1), (2, 6911), (2, 700_001), (3, 450_007), (2, 3_000_000)])
def test_relaxed_sort_is_sorted_permutation(words, n):
    """mhb_sort_records_relaxed (unstable first pass, mhb_part.cuh): ascending on the sorted bytes and a permutation of
    the input - only the order among records with ALL sorted bytes equal may differ from the stable sort"""
    torch = _torch()
    from megahit_b200 import dev
    rng = np.random.default_rng(words * 7 + n)
    recs = rng.integers(0, 2 ** 32, size=(n, words), dtype=np.uint64).astype(np.uint32)
    recs[:, 0] &= np.uint32(0x00FF0F0F)  # long runs of equal keys
    sort_bytes = list(range(1, 4 * words)) if words == 2 else [2, 5, 6, 7, 8, 9, 10, 11]
    a = torch.from_numpy(np.concatenate([recs.view(np.int32).reshape(-1), np.zeros(4, np.int32)])).cuda()
    out = dev.sort_records(a, torch.empty_like(a), n, words, sort_bytes, relaxed=True)
    got = out[: n * words].cpu().numpy().view(np.uint32).reshape(n, words)
    exp = _np_lsd(recs, sort_bytes)

    def key(x):  # the sorted bytes as one comparable integer per record
        v = np.zeros(len(x), dtype=object)
        for b in reversed(sort_bytes):
            v = v * 256 + ((x[:, words - 1 - (b >> 2)] >> np.uint32(8 * (b & 3))) & 255).astype(object)
        return v
    if n <= 800_000:
        assert (key(got) == key(exp)).all()
    full = lambda x: np.sort(np.ascontiguousarray(x).view([("", x.dtype)] * words).reshape(-1))
    assert (full(got) == full(recs)).all()
    # digit-wise check that scales: every sorted byte column of got equals the stable result's
    for b in sort_bytes:
        col = lambda x: (x[:, words - 1 - (b >> 2)] >> np.uint32(8 * (b & 3))) & 255
        assert (col(got) == col(exp)).all()


def test_fused_build_detects_a_rare_odd_length_read_on_the_device():
    """mhb_build_host samples the length words of a library whose size matches a fixed length and lets the device verify
    all of them (mhb_check_fixed_len); a single shorter read outside the sample must send the build through the indexed
    path - same result as the oracle"""
    OP, O = _oracle()
    n_reads, L, k, m = 6000, 150, 27, 2
    b = synth.synth_reads(n_reads, L, 30000, 0.01, seed=77).copy()
    victim = 3333  # not in the first 1024, not a multiple of the sampling step
    b[victim, 0] = 147  # same number of packed words, three bases shorter
    b[victim, 1 + 9] &= np.uint32(0xFC000000)  # bases 144..146 stay, the tail is zero as buildlib leaves it
    reads = O.unpack_bin(b.tobytes(), reverse=True)
    oc = OP.oracle_count(reads, k, m)
    g = lib.build_host(b.reshape(-1), n_reads, k, m, need_mercy=True, want_edges=True)
    assert g["n_solid"] == oc["n_solid"] and (g["edges"] == oc["edges"]).all()
    assert (g["cand_ids"] == oc["cand_ids"]).all()
    seqs, mult = O.edges_as_seqs(oc["edges"], k)
    cand = O.unpack_bin(oc["cand_bytes"], reverse=False)
    me = O.gen_mercy(oc["edges"], cand, k)
    if len(me):
        seqs = O.Seqs.concat([seqs, O.Seqs.from_fixed(me, k + 1)])
        mult = np.concatenate([mult, np.ones(len(me), np.uint16)])
    os_ = O.seq2sdbg(seqs, mult, k)
    assert g["bytes"] == os_["bytes"]
