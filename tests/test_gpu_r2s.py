"""GPU tests of read2sdbg (SURVEY.md 8a A12, the 1-pass route: `megahit --kmin-1pass`, and what the driver runs for
--min-count 1): the CUDA path through the C ABI against

* the fixtures minted by the unmodified reference binary (tests/golden_r2s/r2s.json) - 28 runs: toy set, synthetic
  150 bp reads at k = 21 ... 141 and the reference's k = 255 / min-count 1 case, variable-length reads, poly-A,
  tandem repeats, end-overlapping reads (13 x more mercy than solid edges), and three seeded libraries whose buckets lie
  far above kmsort's insertion-sort threshold, where the reference's result depends on kmsort's order among tied
  records (a stable sort gives other bytes - checked on the oracle, tests/test_oracle_r2s.py);
* the oracle on the intermediate state (solid-edge bits are not visible through the ABI; the SdBG is);
* the reference binary's output at 300 k reads (digests in tests/golden/scale/), through the CLI (`megahit_core read2sdbg`).
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from megahit_b200 import formats as F
from megahit_b200 import lib
from oracle import oracle as O
from oracle import scale_golden as SG
from test_oracle_r2s import R2S, r2s_reads

pytestmark = pytest.mark.gpu

OURS = os.path.join(ROOT, "megahit_b200", "bin", "megahit_core")


def gpu_cases():
    out = []
    for r in R2S["runs"]:
        if r["m"] > 1 and r["k"] > 237:
            continue  # stage-1 records wider than 17 words: forwarded to the reference by the CLI (test below)
        out.append(pytest.param(r, id=f"{r['lib'].split('/')[-1]}-k{r['k']}-m{r['m']}-mercy{r['mercy']}"))
    return out


def n_reads_of(lib_name, data):
    if lib_name.startswith("synth:"):
        return R2S["synth"][lib_name[6:]]["n_reads"]
    return F.read_lib_info(os.path.join(ROOT, "tests", lib_name, "reads.lib"))[1]


@pytest.mark.parametrize("gold", gpu_cases())
def test_read2sdbg_host_matches_reference(gold):
    data = r2s_reads(gold["lib"])
    g = lib.read2sdbg_host(np.frombuffer(data, np.uint32), n_reads_of(gold["lib"], data), gold["k"], gold["m"],
                           bool(gold["mercy"]))
    assert g["n_mercy"] == gold["n_mercy"]
    if gold["m"] > 1:
        assert F.sha256(O.counting_text(g["counting"])) == gold["counting_sha256"]
    assert g["n_items"] == gold["sdbg_items"] and g["n_tips"] == gold["sdbg_tips"]
    assert g["n_large_mul"] == gold["sdbg_large_mul"] and g["words_per_tip_label"] == gold["sdbg_words_per_tip_label"]
    assert F.sha256(lib.sdbg_stream_from_table(g["bucket_table"], g["bytes"])) == gold["sdbg_sha256"]


@pytest.mark.parametrize("env", [{"MHB_R2S_KMSORT_GLOBAL": "1"}, {"MHB_R2S_KM_CAP": "1024"}])
@pytest.mark.parametrize("lib_name", ["synth:deep", "synth:mid", "golden/polya_k27"])
def test_read2sdbg_kmsort_fallback_paths(lib_name, env):
    """the in-place walk on global memory - as the whole sort (MHB_R2S_KMSORT_GLOBAL) and as the per-bucket fall-back of
    the shared-memory form for buckets that exceed the tag capacity of a CTA (forced by a tiny capacity)"""
    gold = [r for r in R2S["runs"] if r["lib"] == lib_name and r["k"] == 27 and r["m"] == 2 and r["mercy"] == 1][0]
    data = r2s_reads(lib_name)
    os.environ.update(env)
    try:
        g = lib.read2sdbg_host(np.frombuffer(data, np.uint32), n_reads_of(lib_name, data), 27, 2, True)
    finally:
        for k_ in env:
            del os.environ[k_]
    assert g["n_mercy"] == gold["n_mercy"] and F.sha256(O.counting_text(g["counting"])) == gold["counting_sha256"]
    assert F.sha256(lib.sdbg_stream_from_table(g["bucket_table"], g["bytes"])) == gold["sdbg_sha256"]


def test_read2sdbg_matches_oracle_tables():
    """bucket table / w counts / ones, which the digests do not cover"""
    data = r2s_reads("golden/syn150_k27")
    reads = O.unpack_bin(data, reverse=True)
    o = O.read2sdbg(reads, 27, 2, True)
    g = lib.read2sdbg_host(np.frombuffer(data, np.uint32), 3000, 27, 2, True)
    assert g["bytes"] == o["bytes"]
    assert (g["bucket_table"][:, 1] == o["bucket_items"]).all() and (g["bucket_table"][:, 2] == o["bucket_tips"]).all()
    nz = o["bucket_items"] > 0
    assert (g["bucket_table"][nz, 0] == o["bucket_byte_off"][:-1][nz]).all()
    assert (g["w_count"] == o["w_count"]).all() and g["ones_in_last"] == o["ones_in_last"]
    assert (g["counting"] == o["counting"]).all()


def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    assert r.returncode == 0, (cmd, r.stderr[-2000:])
    return r


@pytest.mark.parametrize("m,mercy", [(2, True), (1, False)])
def test_cli_read2sdbg_matches_reference_binary_at_300k_reads(tmp_path, m, mercy):
    """the sub-command itself, against what the reference binary wrote for the same seeded library; buckets of ~600
    stage-1 records (kmsort's radix levels decide the tie order), 37 M stage-1 records, 70+ M stage-2 items"""
    libp = str(tmp_path / "reads.lib")
    SG.r2s_lib(libp)
    p = str(tmp_path / "ours")
    _run(SG.r2s_argv(OURS, libp, p, m, mercy, min(32, os.cpu_count() or 8)))
    got = SG.sdbg_digests(p)
    if m > 1:
        got["counting"] = F.file_sha256(p + ".counting")
    assert os.path.exists(p + ".mercy_cand.0")
    assert got == SG.golden()["read2sdbg_300k_k27"][f"m{m}_mercy{int(mercy)}"]


def test_cli_forwards_wide_stage1_to_reference(tmp_path):
    """k = 255 with min count 2: stage-1 records of 19 words are outside the device sort; the CLI hands the command,
    unchanged, to the reference binary (MHB_REFERENCE_CORE) instead of failing.  tests/ref_stand_in.py stands in for
    the reference: it records its command line and writes the SdBG the reference writes for this library."""
    gold = [r for r in R2S["runs"] if r["k"] == 255 and r["m"] == 2][0]
    p = str(tmp_path / "o")
    stand_in = tmp_path / "megahit_core_ref"
    stand_in.write_text(f"#!{sys.executable}\nimport sys\nsys.path.insert(0, {os.path.join(ROOT, 'tests')!r})\n"
                        "import ref_stand_in\nref_stand_in.main(sys.argv)\n")
    stand_in.chmod(0o755)
    args = ["read2sdbg", "-k", "255", "-m", "2", "--host_mem", "3e10", "--output_prefix", p, "--num_cpu_threads", "4",
            "--read_lib_file", os.path.join(ROOT, "tests", gold["lib"], "reads.lib"), "--need_mercy"]
    _run([OURS] + args, env=dict(os.environ, MHB_REFERENCE_CORE=str(stand_in)))
    assert json.load(open(p + ".argv.json")) == [str(stand_in)] + args
    assert F.sha256(F.canonical_sdbg(p)[1]) == gold["sdbg_sha256"]
