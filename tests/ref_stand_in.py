"""Stands in for the reference `megahit_core` where a test checks what the CLI hands to it (MHB_REFERENCE_CORE).

`main(argv)` records the command line it was started with in `<output_prefix>.argv.json` and answers `read2sdbg` with
the oracle's SdBG (pinned against the reference's digests in tests/test_oracle_r2s.py), written in one file as the
reference lays it out: `P.sdbg.0` and the part of `P.sdbg_info` that formats.parse_sdbg_info reads (sdbg_meta.cpp).
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402


def write_sdbg(p, k, r):
    open(p + ".sdbg.0", "wb").write(r["bytes"])
    nz = np.nonzero(r["bucket_items"])[0]
    with open(p + ".sdbg_info", "w") as f:
        f.write(f"k {k}\nwords_per_tip_label {r['words_per_tip_label']}\nnum_buckets {len(nz)}\nnum_files 1\n")
        for b in nz:
            f.write(f"{b} 0 {r['bucket_byte_off'][b]} {r['bucket_items'][b]} {r['bucket_tips'][b]} "
                    f"{r['bucket_large_mul'][b]}\n")


def main(argv):
    def opt(name):
        return argv[argv.index(name) + 1]

    p = opt("--output_prefix")
    json.dump(argv, open(p + ".argv.json", "w"))
    if argv[1] != "read2sdbg":
        raise SystemExit(f"the stand-in answers read2sdbg only, not {argv[1]}")
    k, m = int(opt("-k")), int(opt("-m"))
    reads = O.unpack_bin(open(opt("--read_lib_file") + ".bin", "rb").read(), reverse=True)
    write_sdbg(p, k, O.read2sdbg(reads, k, m, "--need_mercy" in argv))
