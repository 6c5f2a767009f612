#!/usr/bin/env python
"""Per-kernel device times of the count stage (extract + partition passes + solid count) on the bench workload
(10 M x 150 bp synthetic reads, 30x, k = 27, m = 2), from torch.profiler.

    python scripts/count_kernels.py [TREE] [--reads N] [--k K] [--steps S]

TREE (default: this repository) is the source tree whose megahit_b200 package is imported, so that two builds can be
compared kernel by kernel.  Prints one JSON line: mean ms per step of every kernel that ran in the stage, and the mean size of the 16-bit buckets
in each eighth of the bucket ids."""
import argparse
import json
import os
import sys

ap = argparse.ArgumentParser()
ap.add_argument("tree", nargs="?", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--reads", type=int, default=10_000_000)
ap.add_argument("--k", type=int, default=27)
ap.add_argument("--steps", type=int, default=3)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.tree))

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from megahit_b200 import dev, synth  # noqa: E402

n_reads, L, k, m = args.reads, 150, args.k, 2
bin2d = synth.synth_reads_torch(n_reads, L, 5 * n_reads, 0.01, seed=1, device="cuda")
bin_dev = torch.cat([bin2d.reshape(-1), torch.zeros(8, dtype=torch.int32, device="cuda")])
del bin2d
plan = dev.CountPlan(n_reads, L, k, m, "cuda", want_mercy=False)


def stage():
    plan.extract(bin_dev)
    plan.sort()
    plan.count()


for _ in range(2):
    stage()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(args.steps):
        stage()
    torch.cuda.synchronize()
# bucket sizes by bucket id (the order the bucket kernel hands buckets out): mean size of each eighth of the ids
x = plan.a[: 2 * plan.n : 2]
sizes = torch.bincount(((x >> 16) & 0xFFFF).long(), minlength=65536).double()
eighths = [round(float(v), 1) for v in sizes.reshape(8, -1).mean(dim=1).cpu()]
out = {}
for e in prof.key_averages():
    t = getattr(e, "device_time_total", None)
    if t is None:
        t = e.cuda_time_total
    if t > 0:
        out[e.key[:90]] = round(t / 1e3 / args.steps, 3)
print(json.dumps({"tree": os.path.abspath(args.tree), "reads": n_reads, "k": k, "hashed": plan.hashed,
                  "n_solid": int(plan.n_solid_dev[0].item()), "bucket_size_by_id_eighth": eighths, "ms_per_step": dict(sorted(out.items(), key=lambda kv: -kv[1]))}))
