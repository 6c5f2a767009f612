"""GPU tests of the selectable paths (environment switches, forced rounds, widest record templates), each in its own
process so that the switch under test is read at library load.  All of them passed on the round-1 driver run (XPASS) and
are ordinary, strict tests since round 2."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_CHILD = r"""
import json, os, sys
import numpy as np
sys.path.insert(0, %r)
from megahit_b200 import formats as F, lib
case, k, m = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
bin_words = np.fromfile(os.path.join(case, "reads.lib.bin"), np.uint32)
_, n_reads = F.read_lib_info(os.path.join(case, "reads.lib"))
g = lib.build_host(bin_words, n_reads, k, m, need_mercy=True, want_edges=True)
print("RESULT " + json.dumps({"sdbg": F.sha256(lib.sdbg_stream_from_table(g["bucket_table"], g["bytes"])),
                              "edges": F.sha256(g["edges"].tobytes()), "n_items": int(g["n_items"])}))
""" % ROOT


@pytest.mark.parametrize("name,k,m,gold", [c for c in golden_cases() if c.values[0] in ("syn150_k27",)])
def test_fused_build_with_chunked_upload_matches_reference(name, k, m, gold):
    """MHB_H2D_CHUNKS (default 4; here 3 and the single-copy path 1): the library uploaded in pieces, extraction
    overlapping the copies -> same SdBG as the reference"""
    import json
    for chunks in ("3", "1"):
        env = dict(os.environ, MHB_H2D_CHUNKS=chunks)
        p = subprocess.run([sys.executable, "-c", _CHILD, os.path.join(GOLDEN, name), str(k), str(m)], env=env,
                           capture_output=True, text=True, timeout=300)
        line = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")]
        assert line, p.stderr[-800:]
        r = json.loads(line[-1][7:])
        assert r["sdbg"] == gold["sdbg_sha256"] and r["edges"] == gold["edges_sha256"]


_CHILD_S2S = r"""
import json, os, sys
import numpy as np
sys.path.insert(0, %r)
sys.path.insert(0, os.path.join(%r, "tests"))
from megahit_b200 import formats as F, lib
import oracle_pipeline as OP
from oracle import oracle as O
case, k, m, div = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
reads = OP.load_reads(case)
oc = OP.oracle_count(reads, k, m)
seqs, mult = O.edges_as_seqs(oc["edges"], k)
one = lib.s2s_host(seqs.words, seqs.word_off, seqs.len, mult, k)
lib.set_s2s_round_limit(max(1, int(one["n_records"]) // div))
try:
    g = lib.s2s_host(seqs.words, seqs.word_off, seqs.len, mult, k)
    err = None
except lib.MhbError as e:
    g, err = None, str(e)
lib.set_s2s_round_limit(0)
out = {"err": err}
if g is not None:
    out.update(same_bytes=bool(g["bytes"] == one["bytes"]), same_table=bool((g["bucket_table"] == one["bucket_table"]).all()),
               n_items=[int(g["n_items"]), int(one["n_items"])], n_tips=[int(g["n_tips"]), int(one["n_tips"])],
               w=[[int(x) for x in g["w_count"]], [int(x) for x in one["w_count"]]],
               ones=[int(g["ones_in_last"]), int(one["ones_in_last"])])
print("RESULT " + json.dumps(out))
""" % (ROOT, ROOT)


@pytest.mark.parametrize("name,k,m,gold", [c for c in golden_cases() if c.values[0] in ("syn150_k27", "synvar_k31_m1")])
@pytest.mark.parametrize("div", [7])
def test_seq2sdbg_in_rounds_matches_one_pass(name, k, m, gold, div):
    """A13 for seq2sdbg: rounds over leading-byte ranges (forced by capping the items per round) reproduce the item
    stream, the bucket table and the counters of the single pass"""
    import json
    p = subprocess.run([sys.executable, "-c", _CHILD_S2S, os.path.join(GOLDEN, name), str(k), str(m), str(div)],
                       capture_output=True, text=True, timeout=600)
    line = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")]
    assert line, p.stderr[-800:]
    r = json.loads(line[-1][7:])
    if r["err"] is not None:
        assert "more than one round can take" in r["err"]
        return
    assert r["same_bytes"] and r["same_table"]
    assert r["n_items"][0] == r["n_items"][1] and r["n_tips"][0] == r["n_tips"][1]
    assert r["w"][0] == r["w"][1] and r["ones"][0] == r["ones"][1]


def _kmax_cases():
    import json
    base = os.path.join(ROOT, "tests", "golden_kmax")
    out = []
    for name in sorted(os.listdir(base)):
        g = json.load(open(os.path.join(base, name, "golden.json")))
        for k, v in sorted(g["by_k"].items(), key=lambda kv: int(kv[0])):
            out.append(pytest.param(os.path.join(base, name), int(k), g["m"], v, id=f"{name}-k{k}"))
    return out


@pytest.mark.parametrize("case,k,m,gold", _kmax_cases())
def test_fused_build_at_largest_k_matches_reference(case, k, m, gold):
    """k = 255 (17-word records, the reference's kmax) and k = 199: the widest record templates have only been
    exercised by the sort and record-builder tests so far; the fixture is pinned on the CPU (test_oracle_kmax.py)"""
    import json
    env = dict(os.environ)
    env.pop("MHB_H2D_CHUNKS", None)
    p = subprocess.run([sys.executable, "-c", _CHILD, case, str(k), str(m)], env=env, capture_output=True, text=True,
                       timeout=300)
    line = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")]
    assert line, p.stderr[-800:]
    r = json.loads(line[-1][7:])
    assert r["edges"] == gold["edges_sha256"] and r["sdbg"] == gold["sdbg_sha256"] and r["n_items"] == gold["sdbg_items"]
