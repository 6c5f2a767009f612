#!/usr/bin/env python
"""Inputs and reference results of the GPU tests that run at bench scale (1 M and 300 k synthetic reads).

The read libraries are regenerated from their seeds; what the UNMODIFIED reference binary computed for them is kept
in tests/golden/scale/ as digests of the canonical streams (SURVEY.md 8c), so that the GPU tests compare with the
reference without running it.  The `iterate` test also needs the k = 21 contigs and bubbles the reference assembled
from its library; they are stored coded against the seeded genome (a sequence that occurs in the genome becomes
`@<position><strand>`) and decoded byte for byte, checked against the digests of the original files.

    python oracle/scale_golden.py      ->  tests/golden/scale/   (needs oracle/_ref/megahit_core_ref: make -C oracle ref)
"""
from __future__ import annotations

import gzip
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from megahit_b200 import formats as F  # noqa: E402
from megahit_b200 import synth  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "megahit_core_ref")
OUT = os.path.join(ROOT, "tests", "golden", "scale")
ITER_FILES = ("k21.contigs.fa", "k21.bubble_seq.fa")
ASM = ["--min_standalone", "200", "--prune_level", "2", "--merge_len", "20", "--merge_similar", "0.95",
       "--cleaning_rounds", "5", "--disconnect_ratio", "0.1", "--low_local_ratio", "0.2", "--min_depth", "2",
       "--bubble_level", "2", "--max_tip_len", "-1", "--careful_bubble"]
# `assemble` numbers and orders its contigs differently from run to run with several threads; with one the stored
# contigs are reproducible
ASM_THREADS = 1
_COMP = str.maketrans("ACGT", "TGCA")


def golden():
    return json.load(open(os.path.join(OUT, "scale.json")))


# ------------------------------------------------------------------------------------------------
# seeded inputs
# ------------------------------------------------------------------------------------------------
def big_lib(prefix):
    """1 M x 150 bp, 30x, 1 % substitutions (the count / seq2sdbg parity case); returns the `.bin` image"""
    n_reads, L = 1_000_000, 150
    b = synth.synth_reads(n_reads, L, 5 * n_reads, 0.01, seed=4242)
    F.write_lib(prefix, b, n_reads, n_reads * L, L)
    return b


def r2s_lib(prefix):
    """300 k x 150 bp, 30x (read2sdbg): buckets of ~600 stage-1 records"""
    n_reads, L = 300_000, 150
    b = synth.synth_reads(n_reads, L, 5 * n_reads, 0.01, seed=777)
    F.write_lib(prefix, b, n_reads, n_reads * L, L)


def repeat_genome_and_lib(prefix):
    """1.5 Mb genome with three planted repeat families, 300 k x 150 bp reads from it (iterate); returns the genome"""
    rng = np.random.default_rng(11)
    n_reads, L, G = 300_000, 150, 1_500_000
    g = rng.integers(0, 4, G, dtype=np.uint8)
    for rl, copies in ((30, 400), (45, 300), (70, 200)):
        rep = rng.integers(0, 4, rl, dtype=np.uint8)
        for p in rng.choice(G - rl, copies, replace=False):
            g[p:p + rl] = rep
    pos = rng.integers(0, G - L + 1, size=n_reads)
    b = g[pos[:, None] + np.arange(L)[None, :]]
    rc = rng.integers(0, 2, size=n_reads).astype(bool)
    b[rc] = 3 - b[rc][:, ::-1]
    e = rng.random(b.shape) < 0.01
    b[e] = (b[e] + rng.integers(1, 4, size=int(e.sum()), dtype=np.uint8)) & 3
    F.write_lib(prefix, F.pack_reads_fixed(b), n_reads, n_reads * L, L)
    return np.frombuffer(b"ACGT", np.uint8)[g].tobytes().decode()


# ------------------------------------------------------------------------------------------------
# contigs coded against the genome
# ------------------------------------------------------------------------------------------------
def encode_fasta(text, genome):
    out = []
    for line in text.splitlines(keepends=True):
        seq = line.rstrip("\n")
        if line.startswith(">") or not seq:
            out.append(line)
            continue
        i = genome.find(seq)
        if i >= 0:
            out.append(f"@{i}+\n")
            continue
        i = genome.find(seq.translate(_COMP)[::-1])
        out.append(f"@{i}-\n" if i >= 0 else line)
    return gzip.compress("".join(out).encode(), 9, mtime=0)


def write_iter_inputs(d, genome):
    """Writes the reference's k = 21 contigs / bubbles into directory d; returns their paths."""
    g = golden()["iterate_300k"]
    paths = []
    for name in ITER_FILES:
        blob = open(os.path.join(OUT, name + ".coded.gz"), "rb").read()
        lines = gzip.decompress(blob).decode().splitlines(keepends=True)
        text = []
        for j, line in enumerate(lines):
            if line.startswith("@"):
                i, strand = int(line[1:-2]), line[-2]
                n = int(lines[j - 1].rsplit("len=", 1)[1])
                s = genome[i:i + n]
                text.append((s if strand == "+" else s.translate(_COMP)[::-1]) + "\n")
            else:
                text.append(line)
        data = "".join(text).encode()
        assert F.sha256(data) == g["inputs_sha256"][name], f"{name}: decoded contigs differ from the reference's"
        p = os.path.join(d, name)
        open(p, "wb").write(data)
        paths.append(p)
    return paths


# ------------------------------------------------------------------------------------------------
# digests of the canonical streams
# ------------------------------------------------------------------------------------------------
def count_sdbg_digests(p):
    """`count` + `seq2sdbg` outputs under prefix p"""
    info, stream, table = F.canonical_sdbg(p)
    return {"edges": F.sha256(F.canonical_edges(p).tobytes()), "cand": F.file_sha256(p + ".cand"),
            "counting": F.file_sha256(p + ".counting"), "sdbg": F.sha256(stream), "k": info.k,
            "wpt": info.words_per_tip_label, "items": int(table[:, 0].sum()), "tips": int(table[:, 1].sum()),
            "large": int(table[:, 2].sum())}


def sdbg_digests(p):
    info, stream, table = F.canonical_sdbg(p)
    return {"sdbg": F.sha256(stream), "k": info.k, "wpt": info.words_per_tip_label, "items": int(table[:, 0].sum()),
            "tips": int(table[:, 1].sum()), "large": int(table[:, 2].sum())}


def edge_set(prefix):
    """(kmer_size, ascending unique records) of an unsorted `.edges` file pair, as `iterate` writes it"""
    info = open(prefix + ".edges.info").read().split()
    assert info[0] == "kmer_size" and info[10] == "is_sorted" and info[11] == "0" and info[7] == "0"
    W, n = int(info[3]), int(info[9])
    e = np.fromfile(prefix + ".edges.0", np.uint32).reshape(-1, W)
    assert len(e) == n
    u = np.unique(e, axis=0)
    assert len(u) == n
    return int(info[1]), u


def r2s_argv(core, lib, p, m, mercy, threads):
    return ([core, "read2sdbg", "-k", "27", "-m", str(m), "--host_mem", "3e10", "--mem_flag", "1", "--output_prefix", p,
             "--num_cpu_threads", str(threads), "--read_lib_file", lib] + (["--need_mercy"] if mercy else []))


def iterate_argv(core, contigs, bubble, lib, p, step, threads):
    return [core, "iterate", "-c", contigs, "-b", bubble, "-t", str(threads), "-k", "21", "-s", str(step), "-o", p,
            "-r", lib + ".bin"]


# ------------------------------------------------------------------------------------------------
# minting (the reference binary on the host cores)
# ------------------------------------------------------------------------------------------------
def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    if r.returncode != 0:
        raise SystemExit(f"command failed: {' '.join(cmd)}\n{r.stderr[-3000:]}")


def _ref_build(lib, p, k, threads):
    _run([REF, "count", "-k", str(k), "-m", "2", "--host_mem", "3e10", "--mem_flag", "1", "--output_prefix", p,
          "--num_cpu_threads", str(threads), "--read_lib_file", lib])
    _run([REF, "seq2sdbg", "--host_mem", "3e10", "--mem_flag", "1", "--output_prefix", p, "--num_cpu_threads",
          str(threads), "-k", str(k), "--kmer_from", "0", "--input_prefix", p, "--need_mercy"])


def mint():
    threads = min(32, os.cpu_count() or 8)
    os.makedirs(OUT, exist_ok=True)
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        big_lib(f"{tmp}/big")
        _ref_build(f"{tmp}/big", f"{tmp}/big_ref", 27, threads)
        res["count_1m_k27_m2"] = count_sdbg_digests(f"{tmp}/big_ref")

        r2s_lib(f"{tmp}/r2s")
        res["read2sdbg_300k_k27"] = {}
        for m, mercy in ((2, True), (1, False)):
            p = f"{tmp}/r2s_m{m}"
            _run(r2s_argv(REF, f"{tmp}/r2s", p, m, mercy, threads))
            d = sdbg_digests(p)
            if m > 1:
                d["counting"] = F.file_sha256(p + ".counting")
            res["read2sdbg_300k_k27"][f"m{m}_mercy{int(mercy)}"] = d

        genome = repeat_genome_and_lib(f"{tmp}/rep")
        p21 = f"{tmp}/k21"
        _ref_build(f"{tmp}/rep", p21, 21, threads)
        _run([REF, "assemble", "-s", p21, "-o", p21, "-t", str(ASM_THREADS)] + ASM, cwd=tmp)
        it = {"inputs_sha256": {}, "steps": {}}
        for name in ITER_FILES:
            it["inputs_sha256"][name] = F.file_sha256(f"{tmp}/{name}")
            open(os.path.join(OUT, name + ".coded.gz"), "wb").write(encode_fasta(open(f"{tmp}/{name}").read(), genome))
        for step in (8, 20):
            p = f"{tmp}/iter{step}"
            _run(iterate_argv(REF, f"{tmp}/{ITER_FILES[0]}", f"{tmp}/{ITER_FILES[1]}", f"{tmp}/rep", p, step, threads))
            ks, u = edge_set(p)
            it["steps"][str(step)] = {"kmer_size": ks, "n_edges": len(u), "edges_sha256": F.sha256(u.tobytes())}
        res["iterate_300k"] = it
    json.dump(res, open(os.path.join(OUT, "scale.json"), "w"), indent=1, sort_keys=True)
    # the coded contigs must decode to what the reference wrote
    with tempfile.TemporaryDirectory() as tmp:
        write_iter_inputs(tmp, repeat_genome_and_lib(f"{tmp}/rep"))
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    if not os.path.exists(REF):
        raise SystemExit("build oracle/_ref first: make -C oracle ref")
    mint()
