"""GPU tests of `iterate` (SURVEY.md 8f N2): the CUDA path through the C ABI against the sets of iterative edges the
unmodified reference wrote (tests/golden_iter/, chain fixtures), against the oracle, through the CLI, and against what the
reference binary wrote at 300 k reads from contigs it assembled (tests/golden/scale/, oracle/scale_golden.py)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from megahit_b200 import formats as F
from megahit_b200 import lib
from oracle import oracle as O
from oracle import scale_golden as SG
from test_oracle_iter import contig_seqs, iter_cases, iter_inputs

pytestmark = pytest.mark.gpu

OURS = os.path.join(ROOT, "megahit_b200", "bin", "megahit_core")


@pytest.mark.parametrize("step", iter_cases())
def test_iterate_host_matches_reference(step):
    files, data = iter_inputs(step)
    cs = contig_seqs(files)
    reads = O.unpack_bin(data, reverse=False)
    g = lib.iterate_host(cs.words, cs.word_off, cs.len, np.frombuffer(data, np.uint32), reads.n, step["k"], step["step"])
    assert g["n_edges"] == step["n_edges"] and g["edges"].shape[1] == step["words_per_edge"]
    assert F.sha256(g["edges"].tobytes()) == step["edges_sha256"]
    want, aligned = O.iterate(cs, reads, step["k"], step["step"])
    assert (g["edges"] == want).all() and g["n_aligned_reads"] == aligned
    mirror = lib.iterate_host(cs.words, cs.word_off, cs.len, np.frombuffer(data, np.uint32), reads.n, step["k"], step["step"],
                              selftest=True)
    assert g["n_flanks"] == mirror["n_flanks"] and g["n_candidates"] == mirror["n_candidates"]


def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    assert r.returncode == 0, (cmd, r.stderr[-2000:])
    return r


_edge_set = SG.edge_set


def test_cli_iterate_on_fixture(tmp_path):
    step = [s for s in __import__("test_oracle_iter").ITER["steps"] if "chain" not in s and s["k"] == 29][0]
    files, _ = iter_inputs(step)
    p = str(tmp_path / "o")
    _run([OURS, "iterate", "-c", files[0], "-b", files[1], "-t", "4", "-k", "29", "-s", "20", "-o", p, "-r",
          os.path.join(ROOT, "tests", "golden_iter", "reads.lib.bin")])
    ks, u = _edge_set(p)
    assert ks == 49 and F.sha256(u.tobytes()) == step["edges_sha256"]


def test_cli_iterate_matches_reference_binary_at_300k_reads(tmp_path):
    """k = 21 contigs the reference assembled from a repeat-rich synthetic genome, then `iterate` 21 -> 29 and 21 -> 41:
    the same set of edges as the reference binary wrote"""
    libp = str(tmp_path / "reads.lib")
    contigs, bubble = SG.write_iter_inputs(str(tmp_path), SG.repeat_genome_and_lib(libp))
    gold = SG.golden()["iterate_300k"]["steps"]
    for step in (8, 20):
        p = str(tmp_path / f"ours_{step}")
        r = _run(SG.iterate_argv(OURS, contigs, bubble, libp, p, step, min(32, os.cpu_count() or 8)))
        ks, u = _edge_set(p)
        gpu = [l for l in r.stderr.splitlines() if "iterate done" in l]
        print(f"iterate 21+{step}: {len(u)} edges {gpu[-1].split('- ')[-1] if gpu else ''}")
        want = gold[str(step)]
        assert ks == want["kmer_size"] == 21 + step
        assert len(u) == want["n_edges"] > 100 and F.sha256(u.tobytes()) == want["edges_sha256"]
