"""GPU tests against the UNMODIFIED reference:

* bench-scale parity: 1 M synthetic 150 bp reads (123 M edge records; thousands of radix tiles per pass, every CTA of
  the persistent kernels busy) through the file-level commands, compared with the digests of what the reference binary
  writes for the same library (canonical streams, SURVEY.md 8c; tests/golden/scale/, oracle/scale_golden.py) - also
  with the count stage forced into >= 5 rounds and through the fused build;
* downstream acceptance (north_star: "the reference's downstream assemble/local/iterate stages consume it unchanged"):
  the reference's `assemble` run on OUR `.sdbg.*` / `.sdbg_info` gives byte-identical contigs to the same command run
  on the reference-built graph (reader: sdbg/sdbg_raw_content.cpp:18-95, sdbg/sdbg_meta.cpp:24-48), and the reference's
  Python driver (src/megahit) completes a multi-k assembly with our `megahit_core` in its bin directory and produces the
  same final contigs as with the reference core.  These two run the reference binary itself (oracle/_ref/, which
  build() compiles with `make -C oracle ref`).
"""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from megahit_b200 import formats as F
from megahit_b200 import lib, synth
from oracle import scale_golden as SG

pytestmark = pytest.mark.gpu

REF = os.path.join(ROOT, "oracle", "_ref", "megahit_core_ref")
DRIVER = os.path.join(ROOT, "oracle", "_ref", "megahit")
OURS = os.path.join(ROOT, "megahit_b200", "bin", "megahit_core")


def _need_ref():
    if not os.path.exists(REF):
        pytest.fail("oracle/_ref/megahit_core_ref is missing: build() compiles it (make -C oracle ref) from the "
                    "reference sources")


def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    assert r.returncode == 0, (cmd, r.stderr[-2000:])
    return r


def _ref_build(core, lib_prefix, p, k, m, threads=8, mercy=True):
    _run([core, "count", "-k", str(k), "-m", str(m), "--host_mem", "3e10", "--mem_flag", "1", "--output_prefix", p,
          "--num_cpu_threads", str(threads), "--read_lib_file", lib_prefix])
    _run([core, "seq2sdbg", "--host_mem", "3e10", "--mem_flag", "1", "--output_prefix", p, "--num_cpu_threads",
          str(threads), "-k", str(k), "--kmer_from", "0", "--input_prefix", p] + (["--need_mercy"] if mercy else []))


_digests = SG.count_sdbg_digests


@pytest.fixture(scope="module")
def big_case(tmp_path_factory):
    """1 M x 150 bp, 30x, 1 % substitutions; the digests of the reference binary's output for it (k=27, m=2, mercy on)"""
    d = tmp_path_factory.mktemp("big")
    libp = str(d / "reads.lib")
    b = SG.big_lib(libp)
    return {"lib": libp, "bin": b, "n_reads": len(b), "ref": SG.golden()["count_1m_k27_m2"], "dir": d}


def test_bench_scale_file_level_matches_reference_binary(big_case):
    p = str(big_case["dir"] / "ours")
    lib.count_run(big_case["lib"], p, k=27, m=2, host_mem=3e10, num_cpu_threads=8)
    lib.seq2sdbg_run(p, k=27, input_prefix=p, need_mercy=True, host_mem=3e10, num_cpu_threads=8)
    assert _digests(p) == big_case["ref"]


def test_bench_scale_count_in_rounds_matches_reference_binary(big_case):
    """A13: the count stage forced into >= 5 rounds at this size"""
    n_rec = big_case["n_reads"] * (150 - 27)
    p = str(big_case["dir"] / "rounds")
    lib.set_round_limit(n_rec // 6)
    try:
        lib.count_run(big_case["lib"], p, k=27, m=2, host_mem=3e10, num_cpu_threads=8)
    finally:
        lib.set_round_limit(0)
    lib.seq2sdbg_run(p, k=27, input_prefix=p, need_mercy=True, host_mem=3e10, num_cpu_threads=8)
    assert _digests(p) == big_case["ref"]


def test_bench_scale_fused_build_matches_reference_binary(big_case):
    g = lib.build_host(big_case["bin"].reshape(-1), big_case["n_reads"], 27, 2, need_mercy=True, want_edges=True)
    ref = big_case["ref"]
    assert F.sha256(g["edges"].tobytes()) == ref["edges"]
    assert F.sha256(lib.sdbg_stream_from_table(g["bucket_table"], g["bytes"])) == ref["sdbg"]
    assert (int(g["n_items"]), int(g["n_tips"]), int(g["n_large_mul"])) == (ref["items"], ref["tips"], ref["large"])


# ------------------------------------------------------------------------------------------------
# downstream acceptance
# ------------------------------------------------------------------------------------------------
ASM = ["--min_standalone", "300", "--prune_level", "2", "--merge_len", "20", "--merge_similar", "0.95",
       "--cleaning_rounds", "5", "--disconnect_ratio", "0.1", "--low_local_ratio", "0.2", "--min_depth", "2",
       "--bubble_level", "2", "--max_tip_len", "-1", "--careful_bubble"]  # src/megahit:866-899 with its defaults


@pytest.mark.parametrize("name,k", [("toy_k21", 21), ("syn150_k27", 27), ("synvar_k21_m3", 21)])
def test_reference_assemble_consumes_our_sdbg(name, k, tmp_path):
    _need_ref()
    import json
    m = json.load(open(os.path.join(GOLDEN, name, "golden.json")))["m"]
    libp = os.path.join(GOLDEN, name, "reads.lib")
    rp, op = str(tmp_path / "ref"), str(tmp_path / "ours")
    _ref_build(REF, libp, rp, k, m, threads=4)
    _ref_build(OURS, libp, op, k, m, threads=4)          # our executable, same argv
    outs = {}
    for tag, p in (("ref", rp), ("ours", op)):
        cp = str(tmp_path / ("contigs_" + tag))
        r = _run([REF, "assemble", "-s", p, "-o", cp, "-t", "1"] + ASM)
        outs[tag] = {s: open(cp + s, "rb").read() for s in (".contigs.fa", ".addi.fa", ".bubble_seq.fa",
                                                            ".final.contigs.fa", ".contigs.fa.info")}
        assert "FATAL" not in r.stderr
    assert outs["ours"][".contigs.fa"], "no contigs at all: the comparison would be vacuous"
    assert outs["ours"] == outs["ref"]


def test_reference_python_driver_runs_on_our_core(tmp_path):
    """src/megahit (the reference's driver, next to the reference binary as its build places it) with OUR megahit_core
    in its bin directory: checkcpu/kmax probes, count + seq2sdbg on the GPU for every k of the list (k_min from the read
    library with mercy edges, k > k_min from contigs + the iterative edges), `iterate` between the k's on the GPU as well
    (since round 2), everything else forwarded; the final contigs must equal those of the reference core."""
    _need_ref()
    if not os.path.exists(DRIVER):
        pytest.fail("oracle/_ref/megahit (the reference's driver script) is missing: make -C oracle ref")
    b = synth.synth_reads(3000, 150, 15000, 0.01, seed=7)
    fa = tmp_path / "reads.fa"
    with open(fa, "w") as f:
        for i, row in enumerate(b):
            L, w = int(row[0]), row[1:]
            f.write(f">r{i}\n" + "".join("ACGT"[(int(w[j >> 4]) >> (30 - 2 * (j & 15))) & 3] for j in range(L)) + "\n")
    finals = {}
    for tag, core in (("ref", REF), ("ours", OURS)):
        bindir = tmp_path / ("bin_" + tag)
        os.makedirs(bindir)
        shutil.copy(DRIVER, bindir / "megahit")
        os.symlink(core, bindir / "megahit_core")
        out = tmp_path / ("out_" + tag)
        env = dict(os.environ, MHB_REFERENCE_CORE=REF)
        r = subprocess.run([sys.executable, str(bindir / "megahit"), "-r", str(fa), "--k-list", "21,29,39", "-o", str(out),
                            "-t", "2", "--keep-tmp-files"], capture_output=True, text=True, env=env)
        assert r.returncode == 0, r.stderr[-3000:] + open(out / "log").read()[-3000:] if (out / "log").exists() else r.stderr
        finals[tag] = open(out / "final.contigs.fa", "rb").read()
        if tag == "ours":
            log = open(out / "log").read()
            assert "megahit_b200" in log, "the driver's log does not show our core running count/seq2sdbg"
    assert finals["ours"] and finals["ours"] == finals["ref"]


# ------------------------------------------------------------------------------------------------
# several GPUs behind the CLI (C++ driver, one forked worker per GPU; needs >= 2 devices)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k", [("syn150_k27", 27), ("syn150_klist", 59), ("lowcov_k21", 21), ("polya_k27", 27)])
def test_cli_multi_gpu_count_matches_reference(name, k, tmp_path):
    """`megahit_core count --gpus N` (mhb_count_run_multi): per-rank `.edges.<r>` / `.sdbg.<r>` + merged tables whose
    canonical streams equal the reference's digests; the following `seq2sdbg --need_mercy` finds the graph already
    built; the reference's `assemble` reads the N-file SdBG and gives the contigs of the reference-built graph"""
    import json
    n_dev = lib.device_count()
    if n_dev < 2:
        pytest.skip("needs at least 2 GPUs")
    n = min(n_dev, 4)
    gold_all = json.load(open(os.path.join(GOLDEN, name, "golden.json")))
    m, gold = gold_all["m"], gold_all["by_k"][str(k)]
    libp = os.path.join(GOLDEN, name, "reads.lib")
    p = str(tmp_path / "multi")
    r = subprocess.run([OURS, "count", "-k", str(k), "-m", str(m), "--host_mem", "1e9", "--mem_flag", "1", "--output_prefix", p,
                        "--num_cpu_threads", "4", "--read_lib_file", libp, "--gpus", str(n)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert f"{n} GPUs" in r.stderr
    r2 = subprocess.run([OURS, "seq2sdbg", "--host_mem", "1e9", "--mem_flag", "1", "--output_prefix", p, "--num_cpu_threads", "4",
                         "-k", str(k), "--kmer_from", "0", "--input_prefix", p, "--need_mercy"], capture_output=True, text=True)
    assert r2.returncode == 0, r2.stderr[-3000:]
    assert "nothing to do" in r2.stderr
    d = _digests(p)
    assert F.parse_edges_info(p).num_files == n and F.parse_sdbg_info(p).num_files == n
    if gold["n_solid"]:
        assert d["edges"] == gold["edges_sha256"]
    assert d["cand"] == gold["cand_sha256"] and d["counting"] == gold["counting_sha256"]
    assert d["sdbg"] == gold["sdbg_sha256"] and d["items"] == gold["sdbg_items"] and d["tips"] == gold["sdbg_tips"]
    # without --need_mercy the marker does not apply: the ordinary single-GPU seq2sdbg reads the N edge files
    q = str(tmp_path / "nomercy")
    r3 = subprocess.run([OURS, "seq2sdbg", "--host_mem", "1e9", "--mem_flag", "1", "--output_prefix", q, "--num_cpu_threads", "4",
                         "-k", str(k), "--kmer_from", "0", "--input_prefix", p], capture_output=True, text=True)
    assert r3.returncode == 0 and "nothing to do" not in r3.stderr, r3.stderr[-2000:]
    if os.path.exists(REF) and gold["sdbg_items"]:
        rp = str(tmp_path / "ref")
        _ref_build(REF, libp, rp, k, m, threads=4)
        outs = []
        for tag, pre in (("ref", rp), ("ours", p)):
            cp = str(tmp_path / ("contigs_" + tag))
            _run([REF, "assemble", "-s", pre, "-o", cp, "-t", "1"] + ASM)
            outs.append(open(cp + ".contigs.fa", "rb").read())
        assert outs[0] == outs[1]
